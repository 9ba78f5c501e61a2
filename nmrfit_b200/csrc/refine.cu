// K13: one bounded Levenberg-Marquardt iteration per spectrum on the normal equations of K12 (FP64, any axis)
//
// One CTA per spectrum.  It receives the K12 block of the trial it proposed last time (or of the start, on the first
// pass), decides accept or reject against the block it keeps for the current point, updates the damping and the
// status, and proposes the next trial from the current point:
//   frozen   j with H_jj = 0, or at lb with g_j > 0, or at ub with g_j < 0 (g is the gradient of s/2)
//   step     (S H S + lam I) y = -S g over the free parameters, S = diag(H_jj^-1/2), delta = S y; lam * 10 and again
//            while the Cholesky factorisation fails
//   trial    clip(x + delta, lb, ub); frozen parameters are copied, never recomputed
// The scaled system is a packed lower triangle in shared memory (D = 196: 19,306 doubles).  Every element of the
// factor and of the two triangular solves is summed by one thread in index order, so the result depends neither on
// the block size nor on the batch, and there are no atomics but the integer count of running spectra.
//
// K15, tied parameters (DESIGN K15): the same iteration over the d free parameters theta of x = T theta + c.  H, g and
// the box become those of theta (TiedMap below); H and g are projected from the full K12 block element by element as
// the triangle is built, and the trial theta is expanded into the full trial x for the next K12 pass.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <type_traits>
#include "nmrfit_internal.h"
#include "../../include/nmrfit_b200.h"

namespace nmrfit {

namespace {

__device__ __forceinline__ int tri(int i) { return i * (i + 1) / 2; }

// The untied problem: theta = x, the box is [lb, ub].
struct IdentityMap {
    int D;
    __device__ __forceinline__ int d() const { return D; }
    __device__ __forceinline__ int master(int m) const { return m; }
    __device__ __forceinline__ double h(const double* H, int D, int m, int n) const { return H[(size_t)m * D + n]; }
    __device__ __forceinline__ double g(const double* g, int m) const { return g[m]; }
    __device__ __forceinline__ void expand(double* x, int m, double t) const { x[m] = t; }
};

// Tied parameters: group m of theta is its master fm[m] plus the dependents, members mem[off[m] .. off[m+1]) in
// ascending index with scales a (1 for the master) and offsets c.  The projected sums run over the members in that
// order, starting from the first term, without FMA: with the identity map they are H and g exactly.
struct TiedMap {
    const RefineTies& ties; // the kernel's parameter: the map is re-read through it, not kept in registers
    int b, D, nfree;
    __device__ __forceinline__ const int* tis() const { return ties.ints + (size_t)b * (3 * D + 2); }
    __device__ __forceinline__ const double* tds() const { return ties.dbls + (size_t)b * 2 * D; }
    __device__ __forceinline__ int d() const { return nfree; }
    __device__ __forceinline__ int off(int m) const { return tis()[1 + m]; }
    __device__ __forceinline__ int mem(int p) const { return tis()[D + 2 + p]; }
    __device__ __forceinline__ int master(int m) const { return tis()[2 * D + 2 + m]; }
    __device__ double h(const double* H, int, int m, int n) const {   // H_theta[m][n] = sum a_j a_k H_jk
        const double* td = tds();
        double s = 0.0;
        const int p0 = off(m), p1 = off(m + 1), q0 = off(n), q1 = off(n + 1);
        for (int p = p0; p < p1; ++p)
            for (int q = q0; q < q1; ++q) {
                const double t = __dmul_rn(__dmul_rn(td[p], td[q]), H[(size_t)mem(p) * D + mem(q)]);
                s = p == p0 && q == q0 ? t : __dadd_rn(s, t);
            }
        return s;
    }
    __device__ double g(const double* g, int m) const {                 // g_theta[m] = sum a_j g_j
        const int p0 = off(m), p1 = off(m + 1);
        double s = __dmul_rn(tds()[p0], g[mem(p0)]);
        for (int p = p0 + 1; p < p1; ++p) s = __dadd_rn(s, __dmul_rn(tds()[p], g[mem(p)]));
        return s;
    }
    __device__ void expand(double* x, int m, double t) const {         // x_j = a_j t + c_j, rounded twice (no FMA)
        const int j0 = master(m), p1 = off(m + 1);
        for (int p = off(m); p < p1; ++p) {
            const int j = mem(p);
            x[j] = j == j0 ? t : __dadd_rn(__dmul_rn(tds()[p], t), tds()[D + p]);
        }
    }
};

// kTied = false is the untied refinement (nmrfit_ctx_refine); lbs / ubs are then the box of x, else the reduced box
// of theta (first d entries of each spectrum's row).
template <bool kTied>
__global__ void __launch_bounds__(256) refine_step_kernel(const double* __restrict__ trial, double* __restrict__ cur,
                                                          RefineState* __restrict__ state, double* __restrict__ xc,
                                                          double* __restrict__ xt, const double* __restrict__ lbs,
                                                          const double* __restrict__ ubs, int N, int D, int max_iter,
                                                          double xtol, int* __restrict__ active, RefineTies ties) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
    RefineState* st = state + b;
    if (st->status != NMRFIT_REFINE_RUNNING) return;     // finished: trial == current, nothing changes any more
    double* A = smem;                                     // packed lower triangle [n(n+1)/2]
    double* sc = A + tri(D);                              // [D] S of the free parameters
    double* z = sc + D;                                   // [D] right-hand side, then the solution
    int* free_idx = reinterpret_cast<int*>(z + D);        // [D]
    __shared__ int s_nfree;

    const size_t DD = (size_t)D * D, per = 2 * DD + D + 2, cper = DD + D + 1;
    const double* T = trial + (size_t)b * per;            // H [D][D] | M [D][D] | g [D] | ssr [2]
    double* C = cur + (size_t)b * cper;                   // H [D][D] | g [D] | s
    double* x = xc + (size_t)b * D;
    double* xtr = xt + (size_t)b * D;
    const double* lb = lbs + (size_t)b * D;
    const double* ub = ubs + (size_t)b * D;
    const auto map = [&] {
        if constexpr (kTied) return TiedMap{ties, b, D, ties.ints[(size_t)b * (3 * D + 2)]};
        else return IdentityMap{D};
    }();

    int status = NMRFIT_REFINE_RUNNING, passes = st->passes + 1, accepted = st->accepted;
    double lam = st->lam;
    const double s_t = T[2 * DD + D];
    bool take;
    if (passes == 1) {                                    // the pass at the start
        bool bad = false;
        for (size_t k = tid; k < cper; k += nt) bad |= !isfinite(k < DD ? T[k] : T[DD + k]);
        bad = __syncthreads_or(bad);
        take = !bad;
        if (bad) status = NMRFIT_REFINE_NONFINITE;
        lam = 1e-3;
    } else {
        const double s_c = C[DD + D];
        take = isfinite(s_t) && s_t < s_c;
        if (take) {
            // the step actually taken, against each parameter's diagonal noise scale at the point it was built from
            const double dof = (double)(N - map.d());
            if constexpr (kTied) {                        // the projected diagonal, staged: z is free until the solve
                for (int m = tid; m < map.d(); m += nt) z[m] = map.h(C, D, m, m);
                __syncthreads();
            }
            bool small = true;
            for (int m = tid; m < map.d(); m += nt) {
                const int j = map.master(m);
                double h;
                if constexpr (kTied) h = z[m];
                else h = C[(size_t)j * D + j];
                small &= fabs(xtr[j] - x[j]) * sqrt(h * dof / s_c) <= xtol;
            }
            small = __syncthreads_and(small);
            lam = fmax(lam / 10.0, 1e-12);
            accepted += 1;
            if (small) status = NMRFIT_REFINE_CONVERGED;
        } else {
            lam *= 10.0;
            if (lam > 1e16) status = NMRFIT_REFINE_STALLED;
        }
    }
    __syncthreads();                                      // the kept block and x are read
    if (take) {
        for (size_t k = tid; k < cper; k += nt) C[k] = k < DD ? T[k] : T[DD + k];
        if (passes > 1)
            for (int j = tid; j < D; j += nt) x[j] = xtr[j];
    }
    if (status == NMRFIT_REFINE_RUNNING && passes >= max_iter) status = NMRFIT_REFINE_MAX_ITER;
    __syncthreads();

    if (status == NMRFIT_REFINE_RUNNING) {
        const double* H = C;
        const double* g = C + DD;
        if constexpr (kTied) {                            // H_theta_mm and g_theta staged in z and A, in parallel
            for (int m = tid; m < map.d(); m += nt) {
                z[m] = map.h(H, D, m, m);
                A[m] = map.g(g, m);
            }
            __syncthreads();
        }
        if (tid == 0) {
            int n = 0;
            for (int m = 0; m < map.d(); ++m) {
                const int j = map.master(m);
                double h, gm;
                if constexpr (kTied) h = z[m], gm = A[m];
                else h = H[(size_t)j * D + j], gm = g[j];
                const bool frozen = h == 0.0 || (x[j] == lb[m] && gm > 0.0) || (x[j] == ub[m] && gm < 0.0);
                if (!frozen) {
                    free_idx[n] = m;
                    sc[n] = 1.0 / sqrt(h);
                    ++n;
                }
            }
            s_nfree = n;
        }
        __syncthreads();
        const int n = s_nfree;
        for (;;) {
            for (int a = 0; a < n; ++a)
                for (int c = tid; c <= a; c += nt)
                    A[tri(a) + c] = sc[a] * map.h(H, D, free_idx[a], free_idx[c]) * sc[c] + (c == a ? lam : 0.0);
            for (int a = tid; a < n; a += nt) z[a] = -(sc[a] * map.g(g, free_idx[a]));
            __syncthreads();
            // left-looking Cholesky, one column at a time: every thread owns rows of the column
            bool ok = true;
            for (int j = 0; j < n && ok; ++j) {
                const double* Lj = A + tri(j);
                for (int i = j + tid; i < n; i += nt) {
                    double* Li = A + tri(i);
                    double t = Li[j];
                    for (int k = 0; k < j; ++k) t = fma(-Li[k], Lj[k], t);
                    Li[j] = i == j ? sqrt(t) : t;         // sqrt of a negative pivot is NaN: caught below
                }
                __syncthreads();
                const double d = Lj[j];
                ok = d > 0.0 && d < INFINITY;
                if (ok)
                    for (int i = j + 1 + tid; i < n; i += nt) A[tri(i) + j] /= d;
                __syncthreads();
            }
            if (ok) break;
            lam *= 10.0;
            if (lam > 1e16) {
                status = NMRFIT_REFINE_STALLED;
                break;
            }
        }
        if (status == NMRFIT_REFINE_RUNNING) {
            for (int j = 0; j < n; ++j) {                 // L v = z
                const double vj = z[j] / A[tri(j) + j];
                for (int i = j + 1 + tid; i < n; i += nt) z[i] = fma(-A[tri(i) + j], vj, z[i]);
                __syncthreads();
                if (tid == 0) z[j] = vj;
            }
            __syncthreads();
            for (int j = n - 1; j >= 0; --j) {            // L^T y = v
                const double* Lj = A + tri(j);
                const double yj = z[j] / Lj[j];
                for (int i = tid; i < j; i += nt) z[i] = fma(-Lj[i], yj, z[i]);
                __syncthreads();
                if (tid == 0) z[j] = yj;
            }
            __syncthreads();
            for (int j = tid; j < D; j += nt) xtr[j] = x[j];
            __syncthreads();
            for (int a = tid; a < n; a += nt) {
                const int m = free_idx[a];
                map.expand(xtr, m, fmin(fmax(x[map.master(m)] + sc[a] * z[a], lb[m]), ub[m]));
            }
        }
    }
    if (status != NMRFIT_REFINE_RUNNING)
        for (int j = tid; j < D; j += nt) xtr[j] = x[j];
    if (tid == 0) {
        st->lam = lam;
        st->f = sqrt((take || passes == 1 ? s_t : C[DD + D]) / (double)N);
        st->passes = passes;
        st->accepted = accepted;
        st->status = status;
        if (active && status == NMRFIT_REFINE_RUNNING) atomicAdd(active, 1);
    }
}

template <bool kTied>
cudaError_t launch_step(const double* trial, double* cur, RefineState* state, double* xc, double* xt, const double* lb,
                        const double* ub, int B, int N, int D, int max_iter, double xtol, int* active,
                        const RefineTies& ties, cudaStream_t st) {
    static bool attr_set[NMRFIT_MAX_DEVICES] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!attr_set[dev % NMRFIT_MAX_DEVICES]) {
        cudaError_t e = cudaFuncSetAttribute(refine_step_kernel<kTied>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set[dev % NMRFIT_MAX_DEVICES] = true;
    }
    const int threads = std::min(256, (D + 31) / 32 * 32);   // one row of the factor per thread
    refine_step_kernel<kTied><<<B, threads, refine_step_smem(D), st>>>(trial, cur, state, xc, xt, lb, ub, N, D,
                                                                       max_iter, xtol, active, ties);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace

size_t refine_step_smem(int D) { return sizeof(double) * ((size_t)D * (D + 1) / 2 + 2 * (size_t)D) + sizeof(int) * D; }

cudaError_t launch_refine_step(const double* trial, double* cur, RefineState* state, double* xc, double* xt,
                               const double* lb, const double* ub, int B, int N, int D, int max_iter, double xtol,
                               int* active, const RefineTies* ties, cudaStream_t st) {
    if (ties)
        return launch_step<true>(trial, cur, state, xc, xt, lb, ub, B, N, D, max_iter, xtol, active, *ties, st);
    return launch_step<false>(trial, cur, state, xc, xt, lb, ub, B, N, D, max_iter, xtol, active, RefineTies{}, st);
}

}  // namespace nmrfit
