// K1: batched objective  f[b][s] = sqrt(mean_i (weights_i * (V_data_i - V_fit_i))^2)
//
// Replaces, for a whole swarm generation at once, what pyswarm obtains by calling
// the reference's numpy objective once per particle:
//   equations.py:152-212  objective      (RMSE, optional imaginary term :205-209)
//   proc_autophase.py:29-36  ps2         (V_data = u cos(phi_i) - v sin(phi_i), phi_i = p0 + p1*i/N)
//   equations.py:141-147  voigt          (yoff added once per peak)
//
// Mapping: a CTA owns a tile of THREADS*R grid points (held in registers: w, u, v,
// weights) and a tile of up to SP particles of one spectrum.  Per particle the
// per-peak constants are broadcast from shared memory and each thread evaluates
// its R points against every peak; the squared residual is reduced with a fixed
// xor-shuffle tree inside the warp, a fixed-order sum over warps, and (in the
// finalize kernel) a fixed-order sum over point tiles - no atomics, so results
// are bit-reproducible and independent of how particles are sharded over GPUs.
//
// Bound: FP64 pipe issue.  FP64 slots per peak-point (TB = exp-table bits):
//   d, d2, q (3) + rcp (3) + acc (1) + arg (1) + [exp (15 | 9 | 8 | 7) + acc (1) where |s| <= 6.5].
// This kernel serves arbitrary (non-uniform) axes and the fit_im modes; fits on a uniform axis run
// objective_uniform.cu.
#include <cuda_runtime.h>
#include "nmrfit_internal.h"
#include "nmrfit_math.cuh"

namespace nmrfit {

// KK: 0 = real only; 1 = reference semantics (equations.py:199 overwrites I_fit, so
// only the LAST peak's Kramers-Kronig curve is compared); 2 = sum over peaks.
template <int THREADS, int R, int TB, int KK>
__global__ void __launch_bounds__(THREADS)
objective_kernel(ObjArgs a) {
    constexpr int NW = THREADS / 32;
    constexpr int NSUM = KK ? 2 : 1;
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z;
    if (a.frozen && a.frozen[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int P = a.P, N = a.N, D = 4 + 3 * P;
    const int s0 = blockIdx.x * a.sp;          // particle tiles on x (no 65,535 limit), point tiles on y
    const int nsp = min(a.sp, a.S - s0);
    const ObjSmem L(a.sp, P, NW, R, TB, NSUM);
    double* coef = smem + L.coef;
    double2* elo = reinterpret_cast<double2*>(smem + L.elo);
    double2* emid = reinterpret_cast<double2*>(smem + L.emid);
    double* tab = smem + L.tab;
    double* pyoff = smem + L.pyoff;
    double* wpart = smem + L.wpart;

    // ---- this thread's grid points
    const int tile0 = blockIdx.y * (THREADS * R);
    const double* sw = a.spec + (size_t)b * 4 * N;
    double w[R], u[R], v[R], wt[R];
#pragma unroll
    for (int j = 0; j < R; ++j) {
        int i = tile0 + j * THREADS + tid;
        bool ok = i < N;
        w[j] = ok ? sw[i] : 0.0;
        u[j] = ok ? sw[N + i] : 0.0;
        v[j] = ok ? sw[2 * N + i] : 0.0;
        wt[j] = ok ? sw[3 * N + i] : 0.0;     // zero weight: padding contributes nothing
    }

    // ---- per-CTA constants: exp table, per-peak coefficients, phase tables
    if (TB) {
        const double* src = ExpTab<TB>::src();
        for (int i = tid; i < (1 << TB); i += THREADS) tab[i] = src[i];
    }
    const double* xb = a.x + ((size_t)b * a.S + s0) * D;
    for (int idx = tid; idx < nsp * P; idx += THREADS) {
        int sp = idx / P, k = idx - sp * P;
        const double* xs = xb + (size_t)sp * D;
        double r = xs[2], width = xs[4 + 3 * k], loc = xs[5 + 3 * k], area = xs[6 + 3 * k];
        PeakCoef c = make_coef(r, width, loc, area);
        double* o = coef + (sp * P + k) * kCoefStride;
        o[0] = c.loc; o[1] = c.kL2; o[2] = c.aL; o[3] = c.nkG2; o[4] = c.aG;
        double iw = 2.0 / width;
        o[5] = iw; o[6] = iw * kSqrtLn2; o[7] = 0.0;
    }
    {
        const int per = 32 + NW * R;
        for (int idx = tid; idx < nsp * per; idx += THREADS) {
            int sp = idx / per, e = idx - sp * per;
            const double* xs = xb + (size_t)sp * D;
            double p0 = xs[0], p1 = xs[1];
            double ang;
            if (e < 32) {
                ang = (p1 * (double)e) / (double)N;                       // lane offset
            } else {
                int wj = e - 32, wi = wj / R, j = wj - wi * R;
                int ib = tile0 + j * THREADS + wi * 32;                    // first point of warp wi, slot j
                ang = p0 + (p1 * (double)ib) / (double)N;
            }
            double sn, cs;
            sincos(ang, &sn, &cs);
            if (e < 32) elo[sp * 32 + e] = make_double2(cs, sn);
            else emid[sp * (NW * R) + (e - 32)] = make_double2(cs, sn);
        }
        for (int sp = tid; sp < nsp; sp += THREADS) pyoff[sp] = (double)P * xb[(size_t)sp * D + 3];
    }
    __syncthreads();

    // ---- main loop over the particle tile
    for (int sp = 0; sp < nsp; ++sp) {
        const double* cf = coef + sp * P * kCoefStride;
        double acc[R];
        const double py = pyoff[sp];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = py;
        double acci[R];
        if (KK == 2) {
#pragma unroll
            for (int j = 0; j < R; ++j) acci[j] = 0.0;
        }
        for (int k = 0; k < P; ++k) {
            const double2 c01 = *reinterpret_cast<const double2*>(cf + k * kCoefStride);
            const double2 c23 = *reinterpret_cast<const double2*>(cf + k * kCoefStride + 2);
            const double aG = cf[k * kCoefStride + 4];
            const double loc = c01.x, kL2 = c01.y, aL = c23.x, nkG2 = c23.y;
#pragma unroll
            for (int j = 0; j < R; ++j) {
                double d = w[j] - loc;
                double d2 = d * d;
                double q = fma(d2, kL2, 1.0);
                double rq = rcp_pos(q);
                acc[j] = fma(aL, rq, acc[j]);
                // beyond |s| = 6.5 the Gaussian is < 4.5e-19 of its height: below half an ulp of the sum
                const double xg = d2 * nkG2;
                if (xg > -(kGaussCut * kGaussCut)) acc[j] = fma(aG, exp_neg<TB>(xg, tab), acc[j]);
                if (KK == 2) {
                    const double kL = cf[k * kCoefStride + 5], kG = cf[k * kCoefStride + 6];
                    double daw = dawson(d * kG, NMRFIT_DAW_TAB, NMRFIT_DAW_TAIL);
                    acci[j] = fma(aL * (d * kL), rq, acci[j]);
                    acci[j] = fma(aG * kTwoOverSqrtPi, daw, acci[j]);
                }
            }
        }
        // residual against the phase-rotated data
        const double2 el = elo[sp * 32 + lane];
        double ss = 0.0, ssi = 0.0;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const double2 em = emid[sp * (NW * R) + warp * R + j];
            double cr = fma(em.x, el.x, -(em.y * el.y));
            double ci = fma(em.y, el.x, em.x * el.y);
            double vd = fma(u[j], cr, -(v[j] * ci));
            double res = wt[j] * (vd - acc[j]);
            ss = fma(res, res, ss);
            if (KK) {
                double idat = fma(u[j], ci, v[j] * cr);
                double ifit;
                if (KK == 2) {
                    ifit = acci[j];
                } else {
                    const double* cl = cf + (P - 1) * kCoefStride;
                    double d = w[j] - cl[0];
                    double q = fma(d * d, cl[1], 1.0);
                    double daw = dawson(d * cl[6], NMRFIT_DAW_TAB, NMRFIT_DAW_TAIL);
                    ifit = fma(cl[2] * (d * cl[5]), rcp_pos(q), (cl[4] * kTwoOverSqrtPi) * daw);
                }
                double resi = wt[j] * (idat - ifit);
                ssi = fma(resi, resi, ssi);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
            if (KK) ssi += __shfl_xor_sync(0xffffffffu, ssi, o);
        }
        if (lane == 0) {
            wpart[(sp * NW + warp) * NSUM] = ss;
            if (KK) wpart[(sp * NW + warp) * NSUM + 1] = ssi;
        }
    }
    __syncthreads();
    for (int idx = tid; idx < nsp * NSUM; idx += THREADS) {
        int sp = idx / NSUM, c = idx - sp * NSUM;
        double t = 0.0;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) t += wpart[(sp * NW + wi) * NSUM + c];
        a.partials[(((size_t)b * a.S + s0 + sp) * gridDim.y + blockIdx.y) * NSUM + c] = t;
    }
}

// fixed-order sum over point tiles, then sqrt(mean) (equations.py:202, 205-209)
// (nw > 1: partials are per region, [n_tiles][nw]: the regions of a tile first, then the tiles)
__global__ void objective_finalize_kernel(const double* __restrict__ partials, int n_tiles, int nsum,
                                          int N, int S, int B, const int* __restrict__ frozen,
                                          double* __restrict__ f, int nw) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * S) return;
    if (frozen && frozen[idx / S]) return;
    const double* p = partials + (size_t)idx * n_tiles * nw * nsum;
    double sv = 0.0, si = 0.0;
    for (int t = 0; t < n_tiles; ++t) {
        if (nw == 1) {
            sv += p[t * nsum];
            if (nsum == 2) si += p[t * nsum + 1];
        } else {
            double tv = 0.0, ti = 0.0;
            for (int w = 0; w < nw; ++w) {
                tv += p[(t * nw + w) * nsum];
                if (nsum == 2) ti += p[(t * nw + w) * nsum + 1];
            }
            sv += tv;
            si += ti;
        }
    }
    double rm = sqrt(sv / (double)N);
    if (nsum == 2) rm = (rm + sqrt(si / (double)N)) / 2.0;
    f[idx] = rm;
}

// ---- launchers ----------------------------------------------------------------
template <int THREADS, int R, int TB, int KK>
static cudaError_t launch_one(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    cudaError_t e = opt_in_smem<objective_kernel<THREADS, R, TB, KK>>(200 * 1024);
    if (e != cudaSuccess) return e;
    dim3 grid((a.S + p.t.sp - 1) / p.t.sp, p.n_tiles, B);
    objective_kernel<THREADS, R, TB, KK><<<grid, THREADS, p.smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_objective_general(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    return dispatch_geometry<2, 4, 8>(p.t, [&](auto T, auto R) {
        return dispatch_tb(p.t.tb, [&](auto TB) {
            return dispatch<0, 1, 2>(a.kk, [&](auto KK) { return launch_one<T, R, TB, KK>(p, a, B, st); });
        });
    });
}

cudaError_t run_objective_plan(const ObjPlan& p, ObjArgs a, int B, const MoveArgs* mv, double* f, cudaStream_t st,
                               cudaEvent_t ev0, cudaEvent_t evm, cudaEvent_t ev1) {
    a.sp = p.t.sp;
    a.n_tiles = p.n_tiles;
    a.nw = p.t.threads / 32;
    a.sub = p.sub;
    a.tile_major = p.tile_major;
    a.stages = p.t.stages;
    a.gpc = p.gpc;
    a.occ = p.t.occ;
    // the FP64 uniform-axis path times its prepare pass (with the swarm's move folded in) as the first leg; the others
    // move the swarm on their own and leave the first leg empty
    const bool two_pass = p.kernel == OBJ_UNIFORM || p.kernel == OBJ_STREAM;
    cudaError_t e;
    if (ev0) cudaEventRecord(ev0, st);
    if (!two_pass) {
        if (evm) cudaEventRecord(evm, st);
        if (mv && (e = launch_swarm_move(mv->s, mv->rp, mv->rg, mv->generation, st)) != cudaSuccess) return e;
    }
    const bool prepare = p.prep_threads > 0;
    if (prepare && (e = launch_objective_prepare(p, a, B, two_pass ? mv : nullptr, st)) != cudaSuccess) return e;
    if (two_pass && evm) cudaEventRecord(evm, st);
    switch (p.kernel) {
        case OBJ_GENERAL: e = launch_objective_general(p, a, B, st); break;
        case OBJ_UNIFORM: e = launch_objective_uniform(p, a, B, st); break;
        case OBJ_STREAM: e = launch_objective_stream(p, a, B, st); break;
        default: e = launch_objective_f32(p, a, B, st); break;
    }
    if (ev1) cudaEventRecord(ev1, st);
    if (e != cudaSuccess) return e;
    if (f) e = launch_objective_finalize(a.partials, p.n_tiles, p.nsum, a.N, a.S, B, a.frozen, f, st, p.nw);
    count_launches(prepare + 1 + (f ? 1 : 0));
    return e;
}

cudaError_t launch_objective_finalize(const double* partials, int n_tiles, int nsum, int N, int S, int B,
                                      const int* frozen, double* f, cudaStream_t st, int nw) {
    const int total = B * S;
    objective_finalize_kernel<<<(total + 255) / 256, 256, 0, st>>>(partials, n_tiles, nsum, N, S, B, frozen, f, nw);
    return cudaGetLastError();
}

}  // namespace nmrfit
