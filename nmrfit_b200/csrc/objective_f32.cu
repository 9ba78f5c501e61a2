// Opt-in FP32 objective (NMRFIT_FP32): same result definition as objective.cu / objective_uniform.cu
// (reference equations.py:152-212), lineshape arithmetic in single precision.  Contract: <= 1e-5
// relative against the FP64 reference objective on identical particle positions.
//
// What stays in double precision, and why:
//   * d = w - loc (one DADD per near peak and thread): a 0.004 ppm line at 3.4 ppm would lose
//     ulp_f32(3.4)/width = 6e-5 of its shape if the subtraction were done in FP32;
//   * the per-particle constants (objective_prepare_kernel: coefficients, near/far split, far-field
//     polynomial, phase anchors) - computed once per particle, converted on load;
//   * the data side of the residual - phase rotation of (u, v), the subtraction V_data - V_fit, the weight and
//     the sum of squares: near the optimum the residual is the noise (1e-4 of the signal), and forming it
//     from two FP32 numbers of size 1 would cost three of its digits.
// The fitted curve itself - Lorentzian (reciprocals four at a time, one MUFU.RCP), Gaussian (two
// ex2.approx anchors + multiplicative recurrence, skipped beyond 6.5 units of s), far-field polynomial
// (12 FFMA) - is FP32, i.e. carries ~1e-7 of the curve's size.
//
// Two kernels: objective_uniform_f32_kernel mirrors objective_uniform_kernel (uniform axis; TMA bulk
// prologue, regions, near masks); objective_general_f32_kernel takes any axis and evaluates every
// peak at every point (one ex2.approx + one rcp.approx per peak-point: SFU-bound).
#include <cuda_runtime.h>
#include <cstdint>
#include "nmrfit_internal.h"
#include "nmrfit_math.cuh"
#include "uniform_common.cuh"

namespace nmrfit {

__device__ __forceinline__ float rcp_f32(float q) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(q));
    return y;
}
__device__ __forceinline__ float exp_f32(float x) {       // e^x, x <= ~80; flushes to zero below -87
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}

// FP32 twin of peak_span.  t0, s0: offsets of the thread's first point (computed in FP64 by the caller).
template <int R>
__device__ __forceinline__ void peak_span_f32(float t0, float s0, float dT, float aL, float aG, float c2, float thr,
                                              float (&acc)[R]) {
#pragma unroll
    for (int j0 = 0; j0 < R; j0 += 4) {
        const float ta = j0 == 0 ? t0 : fmaf((float)j0, dT, t0);
        const float tb = fmaf((float)(j0 + 1), dT, t0), tc = fmaf((float)(j0 + 2), dT, t0), td = fmaf((float)(j0 + 3), dT, t0);
        // q is clamped: beyond |t| = 3e4 the Lorentzian is < 1e-9 of its height, and the product of four stays finite
        const float qa = fminf(fmaf(ta, ta, 1.f), 1e9f), qb = fminf(fmaf(tb, tb, 1.f), 1e9f);
        const float qc = fminf(fmaf(tc, tc, 1.f), 1e9f), qd = fminf(fmaf(td, td, 1.f), 1e9f);
        const float qab = qa * qb, qcd = qc * qd;
        const float ay = aL * rcp_f32(qab * qcd);
        const float yab = ay * qcd, ycd = ay * qab;
        acc[j0] = fmaf(yab, qb, acc[j0]);
        acc[j0 + 1] = fmaf(yab, qa, acc[j0 + 1]);
        acc[j0 + 2] = fmaf(ycd, qd, acc[j0 + 2]);
        acc[j0 + 3] = fmaf(ycd, qc, acc[j0 + 3]);
    }
    if (fabsf(s0) <= thr) {
        const float hG = dT * 0.83255461115769775635f;
        float g = exp_f32(-(s0 * s0));
        float rho = exp_f32(-(hG * fmaf(2.f, s0, hG)));
#pragma unroll
        for (int j = 0; j < R; ++j) {
            acc[j] = fmaf(aG, g, acc[j]);
            if (j + 1 < R) {
                g *= rho;
                if (j + 2 < R) rho *= c2;
            }
        }
    }
}

template <int THREADS, int R>
__global__ void __launch_bounds__(THREADS, 768 / THREADS)
objective_uniform_f32_kernel(ObjArgs a) {
    constexpr int NW = THREADS / 32;
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z;
    if (a.frozen && a.frozen[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int P = a.P, N = a.N, D = 4 + 3 * P, SP = a.sp;
    const int n_tiles = a.n_tiles, tile = blockIdx.y, NRP = n_tiles * NW;
    const int s0 = blockIdx.x * SP, nsp = min(SP, a.S - s0);
    const F32Smem L(SP, P, THREADS, R);
    double2* suv = reinterpret_cast<double2*>(smem + L.uv);
    double* swt = smem + L.wt;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + L.bar);
    double* wpart = smem + L.wpart;
    const double* coef = smem + L.coef;
    const double* part = smem + L.part;
    const double* farc = smem + L.far;
    const double2* anchor = reinterpret_cast<const double2*>(smem + L.anchor);
    const unsigned* mask = reinterpret_cast<const unsigned*>(smem + L.mask);
    const int MW = L.mw;
    float* coef32 = reinterpret_cast<float*>(smem + L.coef32);
    float* far32 = reinterpret_cast<float*>(smem + L.far32);
    constexpr float H = 16.f * R;

    const int tile0 = tile * (THREADS * R);
    const double* sw = a.spec + (size_t)b * 4 * N;
    const double h = a.grid_h[2 * b], w_ulp = a.grid_h[2 * b + 1];
    const size_t q0 = (size_t)b * a.S + s0;

    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t b_coef = SP * P * 8 * 8, b_part = SP * kPartDoubles * 8, b_far = NW * kFarPoly * 8;
        const uint32_t b_anchor = NW * 2 * 8, b_mask = NW * (MW + 1) * 4;
        mbar_expect_tx(bar, b_coef + b_part + SP * (b_far + b_anchor + b_mask));
        bulk_g2s(smem + L.coef, a.prep_coef + q0 * P * 8, b_coef, bar);
        bulk_g2s(smem + L.part, a.prep_part + q0 * kPartDoubles, b_part, bar);
        for (int sp = 0; sp < SP; ++sp) {
            const size_t rs = (q0 + sp) * NRP + (size_t)tile * NW;
            bulk_g2s(smem + L.far + sp * NW * kFarPoly, a.prep_far + rs * kFarPoly, b_far, bar);
            bulk_g2s(smem + L.anchor + sp * NW * 2, a.prep_anchor + rs * 2, b_anchor, bar);
            bulk_g2s(reinterpret_cast<unsigned*>(smem + L.mask) + sp * NW * (MW + 1), a.prep_mask + rs * (MW + 1), b_mask, bar);
        }
    }
    for (int e = tid; e < THREADS * R; e += THREADS) {
        const int i = tile0 + e;
        const bool ok = i < N;
        const int slot = (e % R) * THREADS + e / R;
        suv[slot] = make_double2(ok ? sw[N + i] : 0.0, ok ? sw[2 * N + i] : 0.0);
        swt[slot] = ok ? sw[3 * N + i] : 0.0;
    }
    const int i_first = tile0 + tid * R;
    const double w_first = i_first < N ? sw[i_first] : fma((double)i_first, h, sw[0]);
    const float xi0 = ((float)(lane * R) - 0.5f * (32 * R - 1)) / H;
    __syncthreads();
    mbar_wait(bar, 0);
    for (int e = tid; e < SP * P; e += THREADS) {          // kL, kG, dT, aL, aG, c2, thr of every (particle, peak)
        const double* c = coef + (size_t)e * 8;
        float* o = coef32 + (size_t)e * 8;
        o[0] = (float)c[1]; o[1] = (float)c[2]; o[2] = (float)c[5]; o[3] = (float)c[3];
        o[4] = (float)c[4]; o[5] = (float)c[7]; o[6] = (float)c[6]; o[7] = 0.f;
    }
    for (int e = tid; e < SP * NW * kFarPoly; e += THREADS) far32[e] = (float)farc[e];
    __syncthreads();

    for (int sp = 0; sp < nsp; ++sp) {
        float acc[R];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = 0.f;
        const double* cf = coef + (size_t)sp * P * 8;
        const double* pt = part + sp * kPartDoubles;
        const unsigned* mk = mask + (size_t)(sp * NW + warp) * (MW + 1);
        for (int wd = 0; wd < MW; ++wd)
        for (unsigned m = mk[wd]; m; m &= m - 1) {
            const int k = wd * 32 + __ffs(m) - 1;
            const float4 f0 = *reinterpret_cast<const float4*>(coef32 + ((size_t)sp * P + k) * 8);       // kL, kG, dT, aL
            const float4 f1 = *reinterpret_cast<const float4*>(coef32 + ((size_t)sp * P + k) * 8 + 4);   // aG, c2, thr, -
            const float d0 = (float)(w_first - cf[k * 8]);       // the subtraction in FP64, one conversion
            peak_span_f32<R>(d0 * f0.x, d0 * f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, acc);
        }
        if (mk[MW]) {
            const float* fc = far32 + (size_t)(sp * NW + warp) * kFarPoly;
            float C[kFarPoly];
#pragma unroll
            for (int n = 0; n < kFarPoly; n += 2) {
                const float2 t = *reinterpret_cast<const float2*>(fc + n);
                C[n] = t.x; C[n + 1] = t.y;
            }
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const float xi = fmaf((float)j, 1.f / H, xi0);
                float p = C[kFarPoly - 1];
#pragma unroll
                for (int n = kFarPoly - 2; n >= 1; --n) p = fmaf(p, xi, C[n]);
                acc[j] = fmaf(p, xi, acc[j] + C[0]);
            }
        }
        if (pt[67] != 0.0) {                               // peaks too narrow for the shortcuts: FP64 exact path
            const double* xs = a.x + (q0 + sp) * D;
            double accd[R];
#pragma unroll
            for (int j = 0; j < R; ++j) accd[j] = 0.0;
            for (int k = 0; k < P; ++k) {
                if (!(cf[k * 8 + 6] < 0.0)) continue;
                const SpanCoef c = make_span_coef(xs[2], xs[4 + 3 * k], xs[5 + 3 * k], xs[6 + 3 * k], h, w_ulp, R);
                peak_exact<R, 0>(sw + i_first, N - i_first, w_first, h, c, nullptr, accd);
            }
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] += (float)accd[j];
        }
        const double2 ew = anchor[sp * NW + warp];
        const double2 el = *reinterpret_cast<const double2*>(pt + 2 * lane);
        const double cd = pt[64], sd = pt[65], py = pt[66];
        double cr = fma(ew.x, el.x, -(ew.y * el.y));
        double ci = fma(ew.y, el.x, ew.x * el.y);
        double ss = 0.0;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const double2 uv = suv[j * THREADS + tid];
            const double wt = swt[j * THREADS + tid];
            const double vd = fma(uv.x, cr, -fma(uv.y, ci, py));
            const double res = wt * (vd - (double)acc[j]);
            ss = fma(res, res, ss);
            if (j + 1 < R) {
                const double c2 = fma(cr, cd, -(ci * sd));
                ci = fma(ci, cd, cr * sd);
                cr = c2;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) wpart[sp * NW + warp] = ss;
    }
    __syncthreads();
    if (tid < nsp) {
        double t = 0.0;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) t += wpart[tid * NW + wi];
        a.partials[(q0 + tid) * n_tiles + tile] = t;
    }
}

// ---- any axis: every peak at every point ------------------------------------------------------------
__global__ void __launch_bounds__(kGenThreads32)
objective_general_f32_kernel(ObjArgs a, int n_tiles) {
    extern __shared__ __align__(16) double smem[];         // [sp][P][4] floats packed: kL, kG, aL, aG ; then loc doubles
    const int b = blockIdx.z;
    if (a.frozen && a.frozen[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = kGenThreads32 / 32, R = kGenR32;
    const int P = a.P, N = a.N, D = 4 + 3 * P;
    const int s0 = blockIdx.x * a.sp, nsp = min(a.sp, a.S - s0);
    double* loc = smem;                                    // [sp][P]
    float4* cf = reinterpret_cast<float4*>(smem + a.sp * P);      // [sp][P]
    double* wpart = smem + a.sp * P + 2 * a.sp * P;        // [sp][NW]
    const int tile0 = blockIdx.y * (kGenThreads32 * R);
    const double* sw = a.spec + (size_t)b * 4 * N;
    double w[R];
    float u[R], v[R], wt[R];
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int i = tile0 + j * kGenThreads32 + tid;
        const bool ok = i < N;
        w[j] = ok ? sw[i] : 0.0;
        u[j] = ok ? (float)sw[N + i] : 0.f;
        v[j] = ok ? (float)sw[2 * N + i] : 0.f;
        wt[j] = ok ? (float)sw[3 * N + i] : 0.f;
    }
    const double* xb = a.x + ((size_t)b * a.S + s0) * D;
    for (int idx = tid; idx < nsp * P; idx += kGenThreads32) {
        const int sp = idx / P, k = idx - sp * P;
        const double* xs = xb + (size_t)sp * D;
        const double r = xs[2], width = xs[4 + 3 * k], area = xs[6 + 3 * k];
        const double iw = 2.0 / width;
        loc[idx] = xs[5 + 3 * k];
        cf[idx] = make_float4((float)iw, (float)(iw * kSqrtLn2), (float)(area * r * (iw / kPi)),
                              (float)(area * (1.0 - r) * (iw * kSqrtLn2OverPi)));
    }
    __syncthreads();
    for (int sp = 0; sp < nsp; ++sp) {
        const double* xs = xb + (size_t)sp * D;
        float acc[R];
        const float py = (float)((double)P * xs[3]);
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = py;
        for (int k = 0; k < P; ++k) {
            const double lc = loc[sp * P + k];
            const float4 c = cf[sp * P + k];
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const float d = (float)(w[j] - lc);
                const float t = d * c.x, s = d * c.y;
                acc[j] = fmaf(c.z, rcp_f32(fminf(fmaf(t, t, 1.f), 1e30f)), acc[j]);
                acc[j] = fmaf(c.w, exp_f32(-(s * s)), acc[j]);
            }
        }
        const double p0 = xs[0], p1 = xs[1];
        float ssf = 0.f;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const int i = tile0 + j * kGenThreads32 + tid;
            float sn, cs;
            sincosf((float)fmod(p0 + (p1 * (double)i) / (double)N, 6.283185307179586), &sn, &cs);
            const float res = wt[j] * (fmaf(u[j], cs, -(v[j] * sn)) - acc[j]);
            ssf = fmaf(res, res, ssf);
        }
        double ss = (double)ssf;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) wpart[sp * NW + warp] = ss;
    }
    __syncthreads();
    if (tid < nsp) {
        double t = 0.0;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) t += wpart[tid * NW + wi];
        a.partials[((size_t)b * a.S + s0 + tid) * n_tiles + blockIdx.y] = t;
    }
}

// ---- launcher ------------------------------------------------------------------------------------
template <int THREADS, int R>
static cudaError_t launch_uniform_f32(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    cudaError_t e = opt_in_smem<objective_uniform_f32_kernel<THREADS, R>>(200 * 1024);
    if (e != cudaSuccess) return e;
    dim3 grid((a.S + p.t.sp - 1) / p.t.sp, p.n_tiles, B);
    objective_uniform_f32_kernel<THREADS, R><<<grid, THREADS, p.smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_objective_f32(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    if (a.kk != 0) return cudaErrorNotSupported;           // fit_im needs the FP64 general kernel
    if (p.kernel == OBJ_F32_UNIFORM)
        return dispatch_geometry<4, 8>(p.t, [&](auto T, auto R) { return launch_uniform_f32<T, R>(p, a, B, st); });
    cudaError_t e = opt_in_smem<objective_general_f32_kernel>(200 * 1024);
    if (e != cudaSuccess) return e;
    dim3 grid((a.S + p.t.sp - 1) / p.t.sp, p.n_tiles, B);
    objective_general_f32_kernel<<<grid, kGenThreads32, p.smem, st>>>(a, p.n_tiles);
    return cudaGetLastError();
}

}  // namespace nmrfit
