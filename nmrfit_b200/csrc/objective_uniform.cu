// K1u: batched objective on a UNIFORM frequency axis (w_i = w_0 + i*h, what np.linspace and
// every spectrometer ppm scale produce) - the kernels a fit normally runs.
//
// Same result definition as objective.cu (reference equations.py:152-212 with ps2,
// proc_autophase.py:29-36, and voigt, equations.py:141-147); different arithmetic (nmrfit_math.cuh):
//   * a thread owns R CONSECUTIVE grid points, so the Gaussian of a peak advances along them by a
//     two-multiply recurrence and only its two anchors need an exponential; beyond 6.5 units of s it
//     is skipped (< 4.5e-19 of its height);
//   * Lorentzian reciprocals are taken four at a time from one reciprocal of the product;
//   * Lorentzians of peaks FAR from a far-field cell (a warp's region of 32*R points, or half / a quarter of it
//     on short axes: far_cells_per_region) are not evaluated peak by peak at all: their Taylor series about the
//     cell's centre are summed into ONE polynomial per (particle, cell) - 12 terms, economised to degree 9 and
//     evaluated by even / odd parts with the cell's mirror lane supplying half of a thread's points, ~7 FP64
//     instructions per point for all far peaks together; only the peaks near the cell (1.5 of 12 on average at
//     BASELINE config 2, 2.2 of 24 at config 4) are evaluated individually.
//
// Two passes per swarm generation:
//   objective_prepare_kernel   a CTA takes a few particles: span coefficients of their peaks, phase tables, and
//                              per region the near-peak masks, the far-field polynomials and the phase
//                              anchor -> a few KB per particle in global memory (with the swarm's move folded in
//                              when a swarm runs; positions in page-locked host memory are read in place);
//   objective_stream_kernel    (objective_stream.cu) the evaluation for all but small particle sets;
//   objective_uniform_kernel   the one-group-per-CTA evaluation: grid (particle groups, point tiles, spectra).  A CTA owns THREADS*R
//                              consecutive points (one region of 32*R per warp) and SP particles.  Its
//                              per-particle constants arrive by TMA bulk copies (cp.async.bulk completing
//                              on an mbarrier) issued by one thread while all threads stage the tile's
//                              (u, v, weights) in shared memory; after that the CTA touches no global
//                              memory until it writes SP partial sums.
// (A persistent variant - one CTA per SM slot looping over groups with double-buffered bulk copies - was
// measured 5-10 % slower at BASELINE config 2: a region's cost depends on how many peaks are near it, the
// same regions for every particle, and the hardware's CTA scheduler balances that better than a static
// assignment of tiles to persistent CTAs.)
//
// The squared residual is reduced by a fixed xor-shuffle tree, a fixed-order sum over the warps of a
// tile and (objective_finalize_kernel) over tiles: no atomics, bit-reproducible, independent of how
// particles or spectra are sharded and of how many CTAs run.
//
// The axis is treated as exactly uniform: the anchor uses the stored w of the thread's first point and
// the other R-1 abscissae are anchor + j*h.  That moves an abscissa by at most one ulp(w) (4.4e-16 ppm
// at w ~ 3.4) against the stored value, i.e. <= 5e-13 relative in a curve value for a 0.004 ppm line.
// Peaks for which that bound (kL * ulp(w)) would exceed 1e-11, and peaks narrower than ~3 grid points,
// are evaluated point by point from the stored w instead (peak_exact).  nmrfit_ctx_set_spectrum only
// enables these kernels when every stored w_i is within 4 ulp of w_0 + i*h; otherwise the general kernel runs.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "nmrfit_internal.h"
#include "nmrfit_math.cuh"
#include "uniform_common.cuh"
#include "uniform_eval.cuh"
#include "swarm_common.cuh"

namespace nmrfit {

// Where particle s of spectrum b keeps its per-region constants (in regions; times sub*12, 2 or mask words each):
// particle-major [B][S][n_tiles*nw] for objective_uniform_kernel, tile-major [B][n_tiles][S][nw] for the streamed
// kernel, whose CTA reads one tile's regions of a whole particle group as ONE contiguous block.
struct RegionDst {
    size_t base, tile_stride;
    int shift, mask;                                       // nw = 4 or 8 regions per tile: region rl = (tile, rl & mask)
    __device__ RegionDst(const ObjArgs& a, int b, int s, int NRP) {
        shift = a.nw == 8 ? 3 : 2;
        mask = a.nw - 1;
        if (a.tile_major) {
            base = ((size_t)b * a.n_tiles * a.S + s) * a.nw;
            tile_stride = (size_t)a.S * a.nw;
        } else {
            base = ((size_t)b * a.S + s) * NRP;
            tile_stride = (size_t)a.nw;
        }
    }
    __device__ size_t region(int rl) const { return base + (size_t)(rl >> shift) * tile_stride + (size_t)(rl & mask); }
};

// ---- pass 1: per-particle constants, once per swarm generation ------------------------------------
// A CTA of kPrepThreads threads takes G consecutive particles of one spectrum and spreads their work items
// (uniform_eval.cuh: span coefficients, phase table, region anchors, then the far-field cells) over all its threads,
// so that every warp is busy in either phase whatever the shape: with one particle per CTA, 6 peaks and 16 regions
// left most lanes idle (r02a: 0.17 ms of a 1.3 ms generation at 6 peaks x 4,096 points x 65,536 particles).
// MOVE: the swarm's move (pso.cu's swarm_move_kernel for these particles) in front: one launch fewer per generation.
// Regions are stored in axis order, padded to a whole number of tiles; the slots of regions past the end of the axis
// are neutral.
template <int R, bool MOVE>
__global__ void __launch_bounds__(kPrepThreads, 4)
objective_prepare_kernel(ObjArgs a, MoveArgs mv, int G) {
    const int nthreads = blockDim.x;
    extern __shared__ __align__(16) double sm[];           // cs [G][P][8], farpk [G][P][4], the (moved) particles [G][D]
    const int b = blockIdx.y, s0 = blockIdx.x * G, tid = threadIdx.x;
    if (MOVE ? mv.s.stop[b] != 0 : (a.frozen && a.frozen[b])) return;
    const int P = a.P, N = a.N, D = 4 + 3 * P, sub = a.sub;
    const int NRP = a.n_tiles * a.nw, nc = NRP * sub, cell_pts = 32 * R / sub;
    const int MWR = mask_words_per_region(P, sub);
    const int ng = min(G, a.S - s0);
    double* cs = sm;
    double* farpk = sm + (size_t)G * P * 8;
    double* xsm = farpk + (size_t)G * P * 4;
    const double* sw = a.spec + (size_t)b * 4 * N;
    const double h = a.grid_h[2 * b], w_ulp = a.grid_h[2 * b + 1];
    const size_t ps0 = (size_t)b * a.S + s0;
    if (MOVE) {
        const SwarmState& s = mv.s;
        const float inv_D = 1.0f / (float)D;
        for (int e = tid; e < ng * D; e += nthreads) {
            const int g = fast_div(e, D, inv_D), d = e - g * D;
            const size_t idx = (ps0 + g) * D + d;
            double rp, rg;
            if (mv.rp) {
                rp = mv.rp[idx];
                rg = mv.rg[idx];
            } else {
                const Philox2 u = philox_uniform2(s.seed, elem_counter(s, b, s0 + g, d), (unsigned long long)mv.generation);
                rp = u.a;
                rg = u.b;
            }
            double x = s.x[idx], v = s.v[idx];
            move_element(s.omega, s.phip, s.phig, rp, rg, s.p[idx], s.g[(size_t)b * D + d], s.lb[(size_t)b * D + d],
                         s.ub[(size_t)b * D + d], x, v);
            s.v[idx] = v;
            s.x[idx] = x;
            xsm[e] = x;
        }
        __syncthreads();
    } else {
        // the positions of the CTA's particles, once, into shared memory (every item below reads them from there).  With
        // x_in they come straight from the caller's page-locked host array - the host-to-device copy happens inside this
        // kernel, overlapped with the other CTAs' arithmetic - and are left in a.x for the evaluation kernel.
        const double* src = (a.x_in ? a.x_in : a.x) + ps0 * D;
        double* keep = a.x_in ? const_cast<double*>(a.x) + ps0 * D : nullptr;
        for (int e = tid; e < ng * D; e += nthreads) {
            const double v = src[e];
            xsm[e] = v;
            if (keep) keep[e] = v;
        }
        __syncthreads();
    }
    // ---- phase 1: per particle kTableItems + NRP rotation items (one sincos each; packed, so that the warps are
    // full whatever the shape) from the first thread up, P span coefficients from the last thread down
    const int per = kTableItems + NRP;
    const float inv_per = 1.0f / (float)per, inv_P = 1.0f / (float)P;
    const double inv_N = 1.0 / (double)N;
    for (int e = tid; e < ng * per; e += nthreads) {
        const int g = fast_div(e, per, inv_per), it = e - g * per;
        const double* xs = xsm + (size_t)g * D;
        double sn, cn;
        sincos(prep_item_angle<R>(xs, it, N, inv_N), &sn, &cn);
        double* dst;
        if (it < kTableItems) {
            dst = a.prep_part + (ps0 + g) * kPartDoubles + 2 * it;
        } else {
            const RegionDst rd(a, b, s0 + g, NRP);
            dst = a.prep_anchor + rd.region(it - kTableItems) * 2;
        }
        *reinterpret_cast<double2*>(dst) = make_double2(cn, sn);
    }
    for (int e = nthreads - 1 - tid; e < ng * P; e += nthreads) {
        const int g = fast_div(e, P, inv_P), k = e - g * P;
        const double* xs = xsm + (size_t)g * D;
        prep_item_coef<R>(xs, k, h, w_ulp, cs + (size_t)g * P * 8, a.prep_coef + (ps0 + g) * P * 8,
                          farpk + (size_t)g * P * 4, sub, P, a.prep_part + (ps0 + g) * kPartDoubles);
    }
    __syncthreads();
    // ---- phase 2: the far-field cells of all ng particles, whole warps (prep_item_cell shuffles)
    for (int e = tid; e < ng; e += nthreads)
        prep_item_exact_count(cs + (size_t)e * P * 8, P, a.prep_part + (ps0 + e) * kPartDoubles);
    const float inv_nc = 1.0f / (float)nc;
    const int sub_shift = sub == 4 ? 2 : sub == 2 ? 1 : 0;
    for (int base = tid & ~31; base < ng * nc; base += nthreads) {
        const int e = base + (tid & 31);
        const bool ok = e < ng * nc;
        const int g = ok ? fast_div(e, nc, inv_nc) : 0, cl = ok ? e - g * nc : 0;
        const int rl = cl >> sub_shift, ci = cl & (sub - 1);  // sub is 1, 2 or 4
        const RegionDst rd(a, b, s0 + g, NRP);
        const size_t rs = rd.region(rl);
        prep_item_cell<R>(ok, cs + (size_t)g * P * 8, farpk + (size_t)g * P * 4, sw, h, N, P, sub, (long long)cl * cell_pts, ci, nullptr,
                          a.prep_far + (rs * sub + ci) * kFarPoly, a.prep_mask + rs * MWR);
    }
}

// ---- pass 2: evaluation ------------------------------------------------------------------------------
template <int THREADS, int R, int TB, int KK>
__global__ void __launch_bounds__(THREADS, (R <= 8 ? 768 : 512) / THREADS)    // 24 (16 for R = 16) resident warps per SM
objective_uniform_kernel(ObjArgs a) {
    constexpr int NSUM = KK ? 2 : 1;
    constexpr int NW = THREADS / 32;
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z;
    if (a.frozen && a.frozen[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int P = a.P, N = a.N, D = 4 + 3 * P, SP = a.sp;
    const int n_tiles = a.n_tiles, tile = blockIdx.y, NRP = n_tiles * NW;
    const int s0 = blockIdx.x * SP, nsp = min(SP, a.S - s0);
    const int SUB = a.sub;
    const UniSmem L(SP, P, THREADS, R, TB, NSUM, SUB);
    double* tab = smem + L.tab;
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
    constexpr double H = 16.0 * R;                         // half a region, in points

    const int tile0 = tile * (THREADS * R);
    const double* sw = a.spec + (size_t)b * 4 * N;
    const double h = a.grid_h[2 * b], w_ulp = a.grid_h[2 * b + 1];
    const size_t q0 = (size_t)b * a.S + s0;                // first particle slot of this group

    // ---- one thread asks the TMA for the group's constants; they complete on the mbarrier.  Whole
    // groups are copied (the prepare buffers are padded), only nsp particles are evaluated.
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const uint32_t b_coef = SP * P * 8 * 8, b_part = SP * kPartDoubles * 8, b_far = NW * SUB * kFarPoly * 8;
        const int MWR = mask_words_per_region(P, SUB);
        const uint32_t b_anchor = NW * 2 * 8, b_mask = NW * MWR * 4;
        mbar_expect_tx(bar, b_coef + b_part + SP * (b_far + b_anchor + b_mask));
        bulk_g2s(smem + L.coef, a.prep_coef + q0 * P * 8, b_coef, bar);
        bulk_g2s(smem + L.part, a.prep_part + q0 * kPartDoubles, b_part, bar);
        for (int sp = 0; sp < SP; ++sp) {
            const size_t rs = (q0 + sp) * NRP + (size_t)tile * NW;
            bulk_g2s(smem + L.far + sp * NW * SUB * kFarPoly, a.prep_far + rs * SUB * kFarPoly, b_far, bar);
            bulk_g2s(smem + L.anchor + sp * NW * 2, a.prep_anchor + rs * 2, b_anchor, bar);
            bulk_g2s(reinterpret_cast<unsigned*>(smem + L.mask) + sp * NW * MWR, a.prep_mask + rs * MWR,
                     b_mask, bar);
        }
    }

    // ---- meanwhile stage the tile: coalesced reads, swizzled [j][thread] placement (uniform_eval.cuh)
    for (int e = tid; e < THREADS * R; e += THREADS) {
        const int i = tile0 + e;
        const bool ok = i < N;
        const int t = e / R, j = e % R;
        const double wgt = ok ? sw[3 * N + i] : 0.0;      // zero weight: padding contributes nothing
        suv[stage_slot_uv(t, j, THREADS)] = stage_point(ok ? sw[N + i] : 0.0, ok ? sw[2 * N + i] : 0.0, wgt);
        swt[stage_slot_wt(t, j, THREADS)] = wgt;
    }
    const int i_first = tile0 + tid * R;                   // this thread's first point
    const double w_first = i_first < N ? sw[i_first] : fma((double)i_first, h, sw[0]);
    if (TB) {
        const double* src = ExpTab<TB>::src();
        for (int i = tid; i < (1 << TB); i += THREADS) tab[i] = src[i];
    }
    const double xi0 = cell_xi0<R>(lane, SUB);             // first point's position inside its far-field cell
    const LaneCell lcell = lane_cell(lane, SUB, P);
    const double inv_H = (double)SUB / H;
    __syncthreads();                                       // tile, table and the mbarrier initialisation are visible
    mbar_wait(bar, 0);                                     // the constants have landed

    // (Assigning the tile's regions to the warps round robin, one particle each, to even out the regions' different
    // costs was measured: no gain - the SM's other CTAs already fill the gaps - and it cost 2 KB of shared memory.)
    for (int sp = 0; sp < nsp; ++sp) {
        double ssi = 0.0;
        const double ss = eval_region<R, TB, KK>(
            coef + (size_t)sp * P * 8, part + sp * kPartDoubles, mask + (size_t)(sp * NW + warp) * mask_words_per_region(P, SUB),
            farc + (size_t)(sp * NW + warp) * SUB * kFarPoly, anchor[sp * NW + warp], MW, P, lane, lcell, w_first, xi0, inv_H,
            suv, swt, tid, THREADS, tab, a.x + (q0 + sp) * D, sw + i_first, N - i_first, h, w_ulp, &ssi);
        if (lane == 0) {
            wpart[(sp * NW + warp) * NSUM] = ss;
            if (KK) wpart[(sp * NW + warp) * NSUM + 1] = ssi;
        }
    }
    __syncthreads();
    for (int idx = tid; idx < nsp * NSUM; idx += THREADS) {
        const int sp = idx / NSUM, c = idx - sp * NSUM;
        double t = 0.0;
#pragma unroll
        for (int wi = 0; wi < NW; ++wi) t += wpart[(sp * NW + wi) * NSUM + c];
        a.partials[((q0 + sp) * n_tiles + tile) * NSUM + c] = t;
    }
}

// ---- launchers ----------------------------------------------------------------
template <int THREADS, int R, int TB, int KK>
static cudaError_t launch_one(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    cudaError_t e = opt_in_smem<objective_uniform_kernel<THREADS, R, TB, KK>>(200 * 1024);
    if (e != cudaSuccess) return e;
    dim3 grid((a.S + p.t.sp - 1) / p.t.sp, p.n_tiles, B);
    objective_uniform_kernel<THREADS, R, TB, KK><<<grid, THREADS, p.smem, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_objective_uniform(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    return dispatch_geometry<4, 8, 16>(p.t, [&](auto T, auto R) {
        return dispatch_tb(p.t.tb, [&](auto TB) {
            return dispatch<0, 1>(a.kk ? 1 : 0, [&](auto KK) { return launch_one<T, R, TB, KK>(p, a, B, st); });
        });
    });
}

// pass 1 (shared with the FP32 evaluation kernel)
cudaError_t launch_objective_prepare(const ObjPlan& p, const ObjArgs& a, int B, const MoveArgs* mv, cudaStream_t st) {
    if (p.t.sp > kPadParticles) return cudaErrorInvalidValue;
    const dim3 grid((a.S + p.prep_g - 1) / p.prep_g, B);
    return dispatch<4, 8, 16>(p.t.r, [&](auto R) {
        if (mv) objective_prepare_kernel<R, true><<<grid, p.prep_threads, p.prep_smem, st>>>(a, *mv, p.prep_g);
        else objective_prepare_kernel<R, false><<<grid, p.prep_threads, p.prep_smem, st>>>(a, MoveArgs{}, p.prep_g);
        return cudaGetLastError();
    });
}

}  // namespace nmrfit
