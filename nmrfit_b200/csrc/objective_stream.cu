// K1s: the STREAMED evaluation kernel of the uniform-axis objective (same result definition and the same
// arithmetic, bit for bit, as objective_uniform.cu: reference equations.py:152-212 with ps2,
// proc_autophase.py:29-36, and voigt, equations.py:141-147; both go through the per-lane steps of uniform_eval.cuh).
//
// What differs is how a CTA is fed.  objective_uniform_kernel gives a CTA one point tile and ONE group of
// particles: stage the tile, wait for the group's constants, evaluate, __syncthreads, write.  ncu (profiles/
// r02a_objective_uniform_metric_full.md and its source page) shows 17 % of all warp samples waiting in that
// frame - 10 % at the final barrier for the CTA's slowest region, 4 % on the constants' mbarrier, 3 % on the tile's
// global loads - with only 24 warps per SM to cover for them.  Here a CTA keeps its tile and walks MANY groups:
//
//   * the tile (u, v, weights and the first abscissa of every thread span) is staged once per CTA;
//   * the groups' per-particle constants stream through a ring of STAGES shared-memory slots filled by TMA bulk
//     copies (cp.async.bulk completing on one mbarrier per slot).  The prepare pass stores the per-region constants
//     tile-major, so a slot is five copies whatever the group size;
//   * a slot is refilled by whichever warp releases it LAST (a ticket in shared memory), so nobody ever waits for a
//     slot to drain: the only waits left are on data that is not there yet;
//   * the CTA's warps take the tile's regions in rotation - group g's region q is evaluated by warp (q - g) mod NW -
//     so every warp sees every region equally often and the regions' different costs (how many peaks are near) no
//     longer make a CTA wait for its slowest warp;
//   * a warp writes its region sums straight to global memory; there is no __syncthreads after the prologue;
//   * with several far-field cells per region (real part, 2 CTAs per SM) a warp evaluates its region for `sub`
//     particles at once, one per group of 32/sub lanes, cell by cell (eval_region_multi): the near peaks of particles
//     in one cell hardly differ - their centres move by a few grid points, the near zone spans a thousand - while the
//     cells of a region often differ by a peak, so the warp visits fewer peaks with idle lanes, and it reads the staged
//     points and reduces once per `sub` particles.
//
// The sums are stored per REGION, partials[B][S][n_tiles][NW]; the finish / finalize kernels add the NW regions of a
// tile first and then the tiles - the order objective_uniform_kernel and the fused swarm kernel use - so the objective
// values are bit-identical across the three.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include "nmrfit_internal.h"
#include "nmrfit_math.cuh"
#include "uniform_common.cuh"
#include "uniform_eval.cuh"

namespace nmrfit {

namespace {

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// OCC: CTAs of 256 threads per SM the kernel is compiled for (3: 80 registers, 75 KB of shared memory each; 2: up to
// 128 registers and 113 KB - room for deeper stages when the per-particle constants are large)
template <int THREADS, int R, int TB, int KK, int OCC, int SUB>
__global__ void __launch_bounds__(THREADS, (R <= 8 ? OCC * 256 : 512) / THREADS)
objective_stream_kernel(ObjArgs a) {
    constexpr int NSUM = KK ? 2 : 1;
    constexpr int NW = THREADS / 32;
    // several particles per warp (eval_region_multi); at 3 CTAs per SM (80 registers) its per-lane particle pointers
    // would spill, so that build keeps one particle per warp
    constexpr bool MULTI = SUB > 1 && !KK && OCC == 2;
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.z;
    if (a.frozen && a.frozen[b]) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int P = a.P, N = a.N, D = 4 + 3 * P, SPG = a.sp, ST = a.stages;
    const int n_tiles = a.n_tiles, tile = blockIdx.y, NRP = n_tiles * NW;
    const StreamSmem L(SPG, ST, P, THREADS, R, TB, SUB);
    const int MW = L.mw;
    double* tab = smem + L.tab;
    double2* suv = reinterpret_cast<double2*>(smem + L.uv);
    double* swt = smem + L.wt;
    double* swf = smem + L.wfirst;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
    int* tickets = reinterpret_cast<int*>(smem + L.tickets);
    double* slots = smem + L.slot0;

    // this CTA's particle groups: [g_lo, g_hi) of the spectrum's ceil(S / SPG)
    const int n_groups = (a.S + SPG - 1) / SPG;
    const int g_lo = blockIdx.x * a.gpc, g_hi = min(n_groups, g_lo + a.gpc);
    const int my_groups = g_hi - g_lo;
    if (my_groups <= 0) return;

    const int tile0 = tile * (THREADS * R);
    const double* sw = a.spec + (size_t)b * 4 * N;
    const double h = a.grid_h[2 * b], w_ulp = a.grid_h[2 * b + 1];
    const size_t pb = (size_t)b * a.S;                     // first particle slot of this spectrum
    const size_t tb_ = ((size_t)b * n_tiles + tile) * a.S; // ... of this (spectrum, tile) in the tile-major arrays

    const uint32_t b_coef = SPG * P * 8 * 8, b_part = SPG * kPartDoubles * 8, b_far = SPG * NW * SUB * kFarPoly * 8;
    const int MWR = mask_words_per_region(P, SUB);
    const uint32_t b_anchor = SPG * NW * 2 * 8, b_mask = SPG * NW * MWR * 4;
    // one thread asks the TMA for group g (relative to g_lo) into slot g % ST.  Whole groups are copied (the
    // prepare buffers are padded); only the particles that exist are evaluated.
    auto fill = [&](int g) {
        const int sl = g % ST;
        double* dst = slots + (size_t)sl * L.slot;
        const size_t q0 = (size_t)(g_lo + g) * SPG;
        uint64_t* bar = bars + sl;
        mbar_expect_tx(bar, b_coef + b_part + b_far + b_anchor + b_mask);
        bulk_g2s(dst + L.coef, a.prep_coef + (pb + q0) * P * 8, b_coef, bar);
        bulk_g2s(dst + L.part, a.prep_part + (pb + q0) * kPartDoubles, b_part, bar);
        bulk_g2s(dst + L.far, a.prep_far + (tb_ + q0) * NW * SUB * kFarPoly, b_far, bar);
        bulk_g2s(dst + L.anchor, a.prep_anchor + (tb_ + q0) * NW * 2, b_anchor, bar);
        bulk_g2s(dst + L.mask, a.prep_mask + (tb_ + q0) * NW * MWR, b_mask, bar);
    };

    if (tid == 0) {
        for (int s = 0; s < ST; ++s) {
            mbar_init(bars + s, 1);
            tickets[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int g = 0; g < min(ST, my_groups); ++g) fill(g);
    }
    // ---- meanwhile stage the tile: coalesced reads, plain [j][thread] placement (uniform_eval.cuh: the stores
    // collide, once per CTA; the evaluation then reads row j of thread t at a compile-time offset from one base)
    for (int e = tid; e < THREADS * R; e += THREADS) {
        const int i = tile0 + e;
        const bool ok = i < N;
        const int t = e / R, j = e % R;
        const double wgt = ok ? sw[3 * N + i] : 0.0;    // zero weight: padding contributes nothing
        suv[j * THREADS + t] = stage_point(ok ? sw[N + i] : 0.0, ok ? sw[2 * N + i] : 0.0, wgt);
        swt[j * THREADS + t] = wgt;
    }
    {
        const int i_first = tile0 + tid * R;
        swf[tid] = i_first < N ? sw[i_first] : fma((double)i_first, h, sw[0]);
    }
    if (TB) {
        const double* src = ExpTab<TB>::src();
        for (int i = tid; i < (1 << TB); i += THREADS) tab[i] = src[i];
    }
    constexpr double H = 16.0 * R;                         // half a region, in points
    const double xi0 = cell_xi0<R>(lane, SUB);             // first point's position inside its far-field cell
    const LaneCell lcell = lane_cell(lane, SUB, P);
    const double inv_H = (double)SUB / H;
    __syncthreads();                                       // the only CTA-wide barrier: tile, table, mbarriers

    // strides between consecutive particles of a slot / of the output
    const int s_coef = P * 8, s_far = NW * SUB * kFarPoly, s_mask = NW * MWR;
    const size_t s_out = (size_t)n_tiles * NW * NSUM;
    int sl = 0;
    uint32_t phase = 0;
    for (int g = 0; g < my_groups; ++g) {
        const double* slot = slots + (size_t)sl * L.slot;
        const size_t q0 = (size_t)(g_lo + g) * SPG;
        const int nsp = min(SPG, a.S - (int)q0);
        // the region of the tile this warp takes for this group (rotation), and the thread span this lane takes
        const int rw = (warp + g) & (NW - 1);
        const int t = rw * 32 + lane;
        const int i_first = tile0 + t * R;
        const double w_first = swf[t];
        const double* cf = slot + L.coef;
        const double* pt = slot + L.part;
        const double* fc = slot + L.far + rw * SUB * kFarPoly;
        const double2* an = reinterpret_cast<const double2*>(slot + L.anchor) + rw;
        const unsigned* mk = reinterpret_cast<const unsigned*>(slot + L.mask) + rw * MWR;
        const double* xs = a.x + (pb + q0) * D;
        double* out = a.partials + (((pb + q0) * n_tiles + tile) * NW + rw) * NSUM;
        mbar_wait(bars + sl, phase);                       // this fill of the slot has landed
        if constexpr (MULTI) {
            // SUB particles per pass over the region, one per 32/SUB-lane group; a short last step repeats the
            // group's last particle in the idle groups and stores nothing for them
            constexpr int LPC = 32 / SUB;
            const int q = lane / LPC;
            for (int sp0 = 0; sp0 < nsp; sp0 += SUB) {
                const int sp = min(sp0 + q, nsp - 1);
                const double ss = eval_region_multi<R, TB, SUB>(
                    cf + sp * s_coef, pt + sp * kPartDoubles, mk + sp * s_mask, fc + sp * s_far, an[sp * NW], MW, P, lane,
                    xi0, inv_H, suv, swt, swf, rw * 32, THREADS, tab, xs + (size_t)sp * D, sw + tile0, N - tile0, h, w_ulp);
                if ((lane & (LPC - 1)) == 0 && sp0 + q < nsp) out[sp * s_out] = ss;
            }
        } else for (int sp = 0; sp < nsp; ++sp) {
            double ssi = 0.0;
            const double ss = eval_region<R, TB, KK, false, SUB>(cf, pt, mk, fc, *an, MW, P, lane, lcell, w_first, xi0, inv_H, suv,
                                                            swt, t, THREADS, tab, xs, sw + i_first, N - i_first, h, w_ulp,
                                                            &ssi);
            if (lane == 0) {
                out[0] = ss;
                if (KK) out[1] = ssi;
            }
            cf += s_coef; pt += kPartDoubles; fc += s_far; an += NW; mk += s_mask; xs += D; out += s_out;
        }
        // release the slot; the warp that releases it last refills it with the group ST further on
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            const int old = atomicAdd(tickets + sl, 1);
            if (old == NW - 1) {
                tickets[sl] = 0;
                __threadfence_block();
                if (g + ST < my_groups) {
                    fence_proxy_async_smem();              // the warps' reads of the slot precede the TMA's writes
                    fill(g + ST);
                }
            }
        }
        if (++sl == ST) { sl = 0; phase ^= 1u; }
    }
    (void)NRP;
}

template <int THREADS, int R, int TB, int KK, int OCC, int SUB>
cudaError_t launch_one(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    cudaError_t e = opt_in_smem<objective_stream_kernel<THREADS, R, TB, KK, OCC, SUB>>(200 * 1024);
    if (e != cudaSuccess) return e;
    const int n_groups = (a.S + p.t.sp - 1) / p.t.sp;
    dim3 grid((n_groups + p.gpc - 1) / p.gpc, p.n_tiles, B);
    objective_stream_kernel<THREADS, R, TB, KK, OCC, SUB><<<grid, THREADS, p.smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace

// Built for the default exp table only (the plan sends every other table to the one-group kernel).  The far-field
// cells per region are a compile-time constant: the lane's cell, the mirror lane and the cell coordinate's step fold
// into immediates instead of being recomputed per particle (the kernel runs at its register limit).
cudaError_t launch_objective_stream(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st) {
    return dispatch_geometry<4, 8, 16>(p.t, [&](auto T, auto R) {
        return dispatch<6>(p.t.tb, [&](auto TB) {
            return dispatch<0, 1>(a.kk ? 1 : 0, [&](auto KK) {
                return dispatch<2, 3>(p.t.occ == 2 ? 2 : 3, [&](auto OCC) {
                    return dispatch<1, 2, 4>(p.sub, [&](auto SUB) { return launch_one<T, R, TB, KK, OCC, SUB>(p, a, B, st); });
                });
            });
        });
    });
}

}  // namespace nmrfit
