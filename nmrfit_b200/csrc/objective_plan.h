// The launch plan of one objective call: which kernel runs, with what geometry, and how much scratch.  Plain C++ with
// no CUDA calls, so that every branch can be checked on the host (tests/test_objective_plan_host.py).
#pragma once
#include <algorithm>
#include <cstddef>
#include "../../include/nmrfit_b200.h"
#include "objective_smem.h"

namespace nmrfit {

struct ObjTune {
    int threads;            // 128 | 256
    int r;                  // grid points per thread: 2 | 4 | 8 (general kernel), 4 | 8 | 16 (uniform-grid kernel)
    int tb;                 // exp table bits: 0 | 6 | 8 | 10
    int sp;                 // particles per CTA (streamed kernel: per pipeline stage)
    int variant;            // uniform-axis FP64 evaluation kernel: 0 one particle group per CTA, 1 streamed (objective_stream.cu)
    int stages;             // streamed kernel: pipeline depth
    int occ;                // streamed kernel: CTAs of 256 threads per SM (2 or 3)
};

constexpr int kPrepThreads = 256;                          // prepare pass: threads per CTA at most

enum ObjKernel {
    OBJ_GENERAL,            // FP64, any axis and every fit_im (objective.cu)
    OBJ_UNIFORM,            // FP64 uniform axis, one particle group per CTA (objective_uniform.cu)
    OBJ_STREAM,             // FP64 uniform axis, streamed particle groups (objective_stream.cu)
    OBJ_F32_UNIFORM,        // FP32 uniform axis (objective_f32.cu)
    OBJ_F32_GENERAL,        // FP32, any axis: 256 threads x 4 points (objective_f32.cu)
};

struct ObjPlan {
    ObjKernel kernel;
    ObjTune t;              // the geometry that runs
    int sub;                // far-field cells per region (1 off the FP64 uniform-axis kernels)
    int n_tiles, nw, nsum;  // partial sums per particle: [n_tiles][nw][nsum] (nw > 1: per region, streamed kernel)
    int tile_major;         // layout of the per-region prepare buffers (streamed kernel)
    int gpc;                // streamed kernel: particle groups per CTA
    int prep_g, prep_threads;   // prepare pass (uniform-axis kernels): particles and threads per CTA; 0 without one
    size_t smem, prep_smem;     // dynamic shared memory of the evaluation kernel and of the prepare pass, bytes
    size_t slots;               // particle slots of the scratch: B*S, or those of the whole particle set a slice is part of
    size_t part_per;            // partial sums per particle slot
    size_t coef, part, far, anchor, mask;   // prepare buffers per particle slot (doubles; mask: 32-bit words) ...
    int pad;                    // ... which hold `pad` slots more: the last group is copied whole
    int refuse;                 // 0, or the NMRFIT_ERR_* code of a refused call ...
    const char* why;            // ... and its message
};

// N points, P peaks, S particles per spectrum, B spectra; `uniform_axis`: every spectrum's w is uniformly spaced;
// `user`: nmrfit_ctx_set_tuning / _set_variant (0 / -1 fields: the library's choice); `far_cells`: 0 or the override
// of far_cells_per_region; `slots_total`: 0, or the particle slots of the whole set when the call evaluates a slice
// of it (nmrfit_objective_batch_host).  The geometry is filled even for a refused call (nmrfit_ctx_get_tuning reports it).
inline ObjPlan objective_plan(int N, int P, int S, int B, int precision, int fit_im, bool uniform_axis, int algorithm,
                              const ObjTune& user, int far_cells, size_t slots_total = 0) {
    ObjPlan p{};
    const bool f32 = precision == NMRFIT_FP32;
    // the uniform-axis kernels (FP64 or FP32) need every spectrum of the batch on a uniform axis and the real-only fit,
    // or in FP64 fit_im with the reference's semantics (last peak's counterpart)
    const bool uni = algorithm != NMRFIT_ALGO_GENERAL && uniform_axis && fit_im != NMRFIT_IM_SUM &&
                     !(fit_im == NMRFIT_IM_REFERENCE && precision != NMRFIT_FP64);
    auto refuse = [&](int code, const char* why) {
        if (!p.refuse) { p.refuse = code; p.why = why; }
    };
    if (algorithm == NMRFIT_ALGO_UNIFORM && !uni)
        refuse(NMRFIT_ERR_STATE, "the uniform-axis kernel needs uniformly spaced w in every spectrum and fit_im off");
    if (f32 && fit_im != NMRFIT_REAL_ONLY)
        refuse(NMRFIT_ERR_ARG, "fit_im is not available in FP32 mode (the Kramers-Kronig term runs in FP64 only)");
    // far-field cells per region of the FP64 uniform-axis kernels (every kernel of a context uses the same split)
    auto cells = [&](int r) { return far_cells ? far_cells : far_cells_per_region(N, r); };
    auto tiles = [&](const ObjTune& g) { return (N + g.threads * g.r - 1) / (g.threads * g.r); };

    ObjTune t;
    // The point tiling fixes the summation order of the residual, so it may depend on
    // N alone (never on how many particles or spectra a rank happens to hold).
    if (uni) {
        // 2,048-point tiles from 2,048 points up (measured 9 % faster than 1,024-point tiles at 2,048 and 4,096
        // points, 6 peaks: tools/tune_probe.py)
        if (N >= 2048) { t.threads = 256; t.r = 8; }
        else { t.threads = 128; t.r = 4; }
    } else {
        if (N >= 8192) { t.threads = 256; t.r = 4; }
        else if (N >= 1024) { t.threads = 128; t.r = 4; }
        else { t.threads = 128; t.r = 2; }
    }
    t.tb = 6;
    if (user.threads) t.threads = user.threads;
    if (user.r) t.r = user.r;
    if (user.tb == -1) t.tb = 0;            // -1: polynomial-only exp
    else if (user.tb > 0) t.tb = user.tb;
    // particles per CTA: amortise the spectrum/coefficients over as many particles as
    // still leaves >= ~4 CTAs per SM
    long long ctas1 = (long long)tiles(t) * S * B;
    int sp = (int)std::max<long long>(1, std::min<long long>(16, ctas1 / (148 * 4)));
    sp = std::min(sp, std::max(1, S));
    if (user.sp > 0) sp = std::min(user.sp, std::max(1, S));
    t.sp = sp;
    // FP64 uniform-axis path: the streamed evaluation kernel (objective_stream.cu) unless the caller asked for the
    // one-group-per-CTA kernel.  Its `sp` is the particles per pipeline stage: as many as leave three CTAs per SM.
    t.variant = 0;
    t.stages = 0;
    t.occ = 3;
    // ... when there is enough work to stream: a small swarm (a single fit's 100-204 particles on a short axis) is a few
    // dozen CTAs either way, and then one group per CTA finishes sooner than a handful of CTAs walking several groups each
    const long long particle_tiles = (long long)tiles(t) * S * B;
    const bool enough = particle_tiles >= 8192 || user.variant == 1;
    bool picked = false;
    if (uni && !f32 && user.variant != 0 && t.tb == 6 && enough) {   // (the streamed kernel is built for the default table)
        t.variant = 1;
        t.occ = user.occ == 3 ? 3 : 2;
        auto stream_bytes = [&]() { return (size_t)StreamSmem(t.sp, t.stages, P, t.threads, t.r, t.tb, cells(t.r)).total * 8; };
        // two CTAs: the B200's 228 KB of shared memory per SM less 1 KB reserved per CTA, halved
        const size_t budget = t.occ == 2 ? 115712 : 74 * 1024;
        // at two CTAs per SM a warp evaluates one particle per far-field cell of a region at once (objective_stream.cu):
        // a group that is not a multiple of that would leave lanes idle in its last step
        const int per_warp = t.occ == 2 ? cells(t.r) : 1;
        auto fit_sp = [&](int stg) {
            t.stages = stg;
            int spg = 0;
            for (int cand = 1; cand <= 16; ++cand) {
                t.sp = cand;
                if (stream_bytes() <= budget && (cand < per_warp || cand % per_warp == 0)) spg = cand;
            }
            return spg;
        };
        int stg = user.stages > 0 ? user.stages : 3;
        int spg = fit_sp(stg);
        // heavy per-particle constants (many peaks, or four far-field cells per region): two deeper stages rather than
        // three shallow ones - a group of 7 instead of 5 particles amortises the per-group handshakes (r02ae: -5 % at
        // 6 peaks x 4,096 points; groups of 7+ gain nothing from the switch)
        if (user.stages == 0 && spg < 6) {
            const int spg2 = fit_sp(2);
            if (spg2 > spg) { stg = 2; spg = spg2; }
        }
        t.stages = stg;
        t.sp = std::max(1, spg);
        bool fits = true;
        if (user.sp > 0) {                                 // an explicit group size: fewer stages if need be, else the
            t.sp = user.sp;                                // one-group-per-CTA kernel below (which takes any size)
            if (stream_bytes() > 200 * 1024 && user.stages == 0) t.stages = 2;
            fits = stream_bytes() <= 200 * 1024;
        }
        if (fits) {
            t.sp = std::min(t.sp, std::max(1, S));
            picked = true;
        } else {
            t.variant = 0;
            t.stages = 0;
            t.occ = 3;
        }
    }
    if (!picked) {
        // per-particle coefficients live in shared memory: keep the CTA under the 200 KB opt-in limit (sized for two
        // sums per point whatever fit_im)
        auto uni_bytes = [&]() {
            return (size_t)(f32 ? F32Smem(t.sp, P, t.threads, t.r).total
                                : UniSmem(t.sp, P, t.threads, t.r, t.tb, 2, cells(t.r)).total) * 8;
        };
        while (t.sp > 1 && (uni ? uni_bytes() : (size_t)ObjSmem(t.sp, P, t.threads / 32, t.r, t.tb, 2).total * 8) > 200 * 1024)
            t.sp /= 2;
        // uniform-axis kernels: three CTAs per SM if a smaller particle tile achieves it (227 KB / 3)
        if (uni && user.sp <= 0)
            while (t.sp > 4 && uni_bytes() > 74 * 1024) t.sp -= 1;
    }
    if (uni && f32 && t.r == 16) t.r = 8;                  // the FP32 kernel is built for 4 and 8
    if (uni ? (t.r != 4 && t.r != 8 && t.r != 16) : (t.r != 2 && t.r != 4 && t.r != 8))
        refuse(NMRFIT_ERR_ARG, uni ? "points_per_thread must be 4, 8 or 16 for the uniform-axis kernel"
                                   : "points_per_thread must be 2, 4 or 8 for the general kernel");

    // scratch: partials sized for two sums per tile of this geometry (and per region when streamed)
    p.slots = std::max((size_t)B * S, slots_total);
    p.part_per = (size_t)tiles(t) * 2 * (t.variant == 1 ? t.threads / 32 : 1);
    p.kernel = f32 ? (uni ? OBJ_F32_UNIFORM : OBJ_F32_GENERAL) : !uni ? OBJ_GENERAL : t.variant == 1 ? OBJ_STREAM : OBJ_UNIFORM;
    if (p.kernel == OBJ_F32_GENERAL) { t.threads = kGenThreads32; t.r = kGenR32; }
    p.t = t;
    p.sub = uni && !f32 ? cells(t.r) : 1;
    p.n_tiles = tiles(t);
    p.nw = p.kernel == OBJ_STREAM ? t.threads / 32 : 1;
    p.nsum = !f32 && fit_im ? 2 : 1;
    p.tile_major = p.kernel == OBJ_STREAM;
    switch (p.kernel) {
        case OBJ_GENERAL: p.smem = (size_t)ObjSmem(t.sp, P, t.threads / 32, t.r, t.tb, p.nsum).total * 8; break;
        case OBJ_UNIFORM: p.smem = (size_t)UniSmem(t.sp, P, t.threads, t.r, t.tb, p.nsum, p.sub).total * 8; break;
        case OBJ_STREAM: p.smem = (size_t)StreamSmem(t.sp, t.stages, P, t.threads, t.r, t.tb, p.sub).total * 8; break;
        case OBJ_F32_UNIFORM: p.smem = (size_t)F32Smem(t.sp, P, t.threads, t.r).total * 8; break;
        case OBJ_F32_GENERAL: p.smem = (size_t)f32_general_smem_doubles(t.sp, P) * 8; break;
    }
    if (p.kernel == OBJ_STREAM) {
        // groups per CTA: enough CTAs for ~5 waves of the 3-per-SM residency (the hardware's CTA scheduler evens out
        // the tiles' different costs), few enough that the tile staging is amortised over >= 4 groups
        const long long n_groups = (S + t.sp - 1) / t.sp;
        long long gpc = n_groups * p.n_tiles * B / (148 * 3 * 5);
        gpc = std::max<long long>(4, std::min<long long>(32, gpc));
        const long long chunks = (n_groups + gpc - 1) / gpc;
        p.gpc = (int)((n_groups + chunks - 1) / chunks);   // equal chunks
    }
    if (uni) {
        // the prepare pass: per-particle constants, per region of a tile (prep_far / prep_anchor / prep_mask)
        const int nc = p.n_tiles * (t.threads / 32) * p.sub;
        p.coef = (size_t)P * 8;
        p.part = kPartDoubles;
        p.far = (size_t)nc * kFarPoly;
        p.anchor = (size_t)p.n_tiles * (t.threads / 32) * 2;
        p.mask = (size_t)p.n_tiles * (t.threads / 32) * mask_words_per_region(P, p.sub);
        p.pad = kPadParticles;
        // particles per CTA: about four rounds of far-field cells for its 256 threads (0.184 / 0.182 / 0.179 ms with
        // 8 / 12 / 16 particles at 6 peaks x 4,096 points; 0.202 with 4)
        const size_t per_particle = (size_t)(P * 12 + 4 + 3 * P) * sizeof(double);
        int G = std::max(1, std::min(16, std::min(S, 4 * kPrepThreads / nc)));
        while (G > 1 && G * per_particle > 40 * 1024) --G; // stay inside the default dynamic shared-memory limit
        // a particle with >= 128 cells fills a CTA of 128 threads on its own (and many small CTAs schedule better)
        int threads = nc >= 128 ? 128 : kPrepThreads;
        if (nc >= 128) G = 1;
        // a small swarm (a single fit): as many CTAs as there are particles - the critical path of one CTA, not the
        // machine's throughput, is what the generation waits for
        const long long want_ctas = 2 * 148;
        if ((long long)S * B / G < want_ctas) {
            G = (int)std::max<long long>(1, std::min<long long>(G, (long long)S * B / want_ctas));
            if (G == 1) threads = 128;
        }
        p.prep_g = G;
        p.prep_threads = threads;
        p.prep_smem = G * per_particle;
    }
    return p;
}

}  // namespace nmrfit
