// Storage layout of the objective kernels: the per-particle constants of the uniform-axis prepare pass and the
// shared-memory carve-up of every evaluation kernel.  Plain C++: the kernels and the launch plan (objective_plan.h,
// compiled for the host as well) size the same memory from the same code.
#pragma once

#ifdef __CUDACC__
#define NMRFIT_HOST_DEVICE __host__ __device__
#else
#define NMRFIT_HOST_DEVICE
#endif

namespace nmrfit {

constexpr int kCoefStride = 8;     // general kernel, per peak: loc kL2 aL nkG2 | aG kL kG pad
constexpr int kPartDoubles = 68;   // per particle: e^{i p1 lane R/N} for 32 lanes (64), cos/sin(p1/N), P*yoff, #exact peaks
constexpr int kPadParticles = 64;  // slack at the end of the prepare buffers: the last group is copied whole
constexpr int kFarPoly = 10;       // coefficients stored per far-field cell (nmrfit_math.cuh: far_economise)

// Far-field cells per warp region (uniform_eval.cuh): the shorter the axis, the shorter the cells, down to 64 points.
// A function of the axis length and the points per thread ONLY, so that every kernel that evaluates a given spectrum
// (one group per CTA, streamed, fused swarm) splits it the same way and stays bit-identical to the others.
NMRFIT_HOST_DEVICE inline int far_cells_per_region(int N, int R) {
    const int target = N < 8192 ? 64 : (N < 32768 ? 128 : 256);    // cell length aimed at, in points
    int sub = 32 * R / target;
    return sub < 1 ? 1 : (sub > 4 ? 4 : sub);
}

// 32-bit mask words per region: one cell - [MW near words][has-far]; several cells - the same block for the UNION of
// the region's cells first (what the warp as a whole has to visit), then one block per cell.
NMRFIT_HOST_DEVICE inline int mask_words_per_region(int P, int sub) { return (sub == 1 ? 1 : sub + 1) * ((P + 31) / 32 + 1); }

// ---- shared-memory carve-ups (in doubles) -------------------------------------------------------------

// general kernel (objective.cu)
struct ObjSmem {
    int coef, pyoff, elo, emid, wpart, tab, total;
    NMRFIT_HOST_DEVICE ObjSmem(int sp, int P, int nwarps, int R, int TB, int nsum) {
        int o = 0;
        coef = o;  o += sp * P * kCoefStride;
        elo = o;   o += sp * 32 * 2;
        emid = o;  o += sp * nwarps * R * 2;
        tab = o;   o += TB ? (1 << TB) : 0;
        pyoff = o; o += sp;
        wpart = o; o += sp * nwarps * nsum;
        total = o;
    }
};

// one-group-per-CTA uniform-axis kernel (objective_uniform.cu); every offset is even (16-byte alignment)
struct UniSmem {
    int tab, uv, wt, bar, wpart, coef, part, far, anchor, mask, mw, total;
    NMRFIT_HOST_DEVICE UniSmem(int sp, int P, int threads, int R, int TB, int nsum = 1, int sub = 1) {
        const int nw = threads / 32;
        mw = (P + 31) / 32;                               // near-peak mask words per region, + 1 has-far word
        int o = 0;
        tab = o;    o += TB ? (1 << TB) : 0;
        uv = o;     o += threads * R * 2;
        wt = o;     o += threads * R;
        bar = o;    o += 2;                               // one mbarrier
        wpart = o;  o += sp * nw * nsum;                   // nsum = 2: real and imaginary sums of fit_im
        coef = o;   o += sp * P * 8;
        part = o;   o += sp * kPartDoubles;
        far = o;    o += sp * nw * sub * kFarPoly;       // far-field polynomial per (particle, cell of a warp region)
        anchor = o; o += sp * nw * 2;                     // phase at the first point of each warp region
        mask = o;   o += ((sp * nw * mask_words_per_region(P, sub) + 3) / 4) * 2;
        total = o;
    }
};

// streamed uniform-axis kernel (objective_stream.cu); every offset is even (16-byte alignment)
struct StreamSmem {
    int tab, uv, wt, wfirst, bars, tickets, slot0, slot, coef, part, far, anchor, mask, mw, total;
    NMRFIT_HOST_DEVICE StreamSmem(int spg, int stages, int P, int threads, int R, int TB, int sub) {
        const int nw = threads / 32;
        mw = (P + 31) / 32;
        int o = 0;
        tab = o;     o += TB ? (1 << TB) : 0;
        uv = o;      o += threads * R * 2;
        wt = o;      o += threads * R;
        wfirst = o;  o += threads;                          // stored abscissa of every thread span's first point
        bars = o;    o += stages;                           // one mbarrier per slot
        tickets = o; o += (stages + 1) / 2 * 2;             // one 32-bit release counter per slot (two per double)
        if (o & 1) ++o;
        slot0 = o;
        // one slot (offsets relative to its start)
        int q = 0;
        coef = q;    q += spg * P * 8;
        part = q;    q += spg * kPartDoubles;
        far = q;     q += spg * nw * sub * kFarPoly;       // per far-field cell (uniform_eval.cuh)
        anchor = q;  q += spg * nw * 2;
        mask = q;    q += ((spg * nw * mask_words_per_region(P, sub) + 3) / 4) * 2;
        slot = q;
        total = slot0 + stages * slot;
    }
};

// FP32 uniform-axis kernel (objective_f32.cu): as UniSmem without the exp table
struct F32Smem {
    int uv, wt, bar, wpart, coef, part, far, anchor, mask, coef32, far32, mw, total;
    NMRFIT_HOST_DEVICE F32Smem(int sp, int P, int threads, int R) {
        const int nw = threads / 32;
        mw = (P + 31) / 32;
        int o = 0;
        uv = o;     o += threads * R * 2;
        wt = o;     o += threads * R;
        bar = o;    o += 2;
        wpart = o;  o += sp * nw;
        coef = o;   o += sp * P * 8;
        part = o;   o += sp * kPartDoubles;
        far = o;    o += sp * nw * kFarPoly;
        anchor = o; o += sp * nw * 2;
        mask = o;   o += ((sp * nw * (mw + 1) + 3) / 4) * 2;
        // single-precision copies made once per CTA (a double -> float conversion costs four FP64 issue slots: doing
        // it per thread and particle was 30 conversions per 8 points, now 1.5 + the 8 of the residual)
        coef32 = o; o += sp * P * 4;                       // 8 floats per peak: kL, kG, dT, aL, aG, c2, thr, -
        far32 = o;  o += (sp * nw * kFarPoly + 1) / 2;
        o = (o + 1) & ~1;
        total = o;
    }
};

// FP32 kernel for any axis (objective_f32.cu): a fixed geometry; [sp][P] locations, [sp][P] float4 coefficients,
// [sp][warps] partial sums
constexpr int kGenThreads32 = 256;
constexpr int kGenR32 = 4;
inline int f32_general_smem_doubles(int sp, int P) { return sp * P * 3 + sp * (kGenThreads32 / 32); }

}  // namespace nmrfit
