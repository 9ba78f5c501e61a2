// Plan equivalence: objective_plan (nmrfit_b200/csrc/objective_plan.h) against the launch decisions it replaced -
// pick_tune, use_uniform and ctx_cells of cabi.cu, the geometry run_objective derived from them, and what the
// launchers of objective.cu, objective_uniform.cu, objective_stream.cu and objective_f32.cu derived in turn - copied
// below from the commit before the plan existed.  Every output field is compared over a grid of shapes and every value
// of the tuning knobs; the summary goes to stdout (profiles/objective_plan_equiv.txt).
//
//     g++ -O2 -std=c++17 -fopenmp -o /tmp/objective_plan_equiv tools/objective_plan_equiv.cpp && /tmp/objective_plan_equiv
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>
#include "../nmrfit_b200/csrc/objective_plan.h"

// the particles-per-CTA values of the sweep (-DSP_VALUES=...; every value by default)
#ifndef SP_VALUES
#define SP_VALUES 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, \
    29, 30, 31, 32, 33, 34, 35, 36, 37, 38, 39, 40, 41, 42, 43, 44, 45, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, \
    58, 59, 60, 61, 62, 63, 64
#define SP_NAME "0..64"
#endif

namespace parent {
using nmrfit::kPartDoubles;
using nmrfit::kPadParticles;
using nmrfit::kFarPoly;
using nmrfit::ObjTune;
constexpr int kCoefStride = 8;
inline int far_cells_per_region(int N, int R) {
    const int target = N < 8192 ? 64 : (N < 32768 ? 128 : 256);
    int sub = 32 * R / target;
    return sub < 1 ? 1 : (sub > 4 ? 4 : sub);
}
inline int mask_words_per_region(int P, int sub) { return (sub == 1 ? 1 : sub + 1) * ((P + 31) / 32 + 1); }

// ---- the carve-ups as the kernel files had them
struct ObjSmem {
    int coef, pyoff, elo, emid, wpart, tab, total;
    ObjSmem(int sp, int P, int nwarps, int R, int TB, int nsum) {
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
struct UniSmem {
    int tab, uv, wt, bar, wpart, coef, part, far, anchor, mask, mw, total;
    UniSmem(int sp, int P, int threads, int R, int TB, int nsum = 1, int sub = 1) {
        const int nw = threads / 32;
        mw = (P + 31) / 32;
        int o = 0;
        tab = o;    o += TB ? (1 << TB) : 0;
        uv = o;     o += threads * R * 2;
        wt = o;     o += threads * R;
        bar = o;    o += 2;
        wpart = o;  o += sp * nw * nsum;
        coef = o;   o += sp * P * 8;
        part = o;   o += sp * kPartDoubles;
        far = o;    o += sp * nw * sub * kFarPoly;
        anchor = o; o += sp * nw * 2;
        mask = o;   o += ((sp * nw * mask_words_per_region(P, sub) + 3) / 4) * 2;
        total = o;
    }
};
struct StreamSmem {
    int tab, uv, wt, wfirst, bars, tickets, slot0, slot, coef, part, far, anchor, mask, mw, total;
    StreamSmem(int spg, int stages, int P, int threads, int R, int TB, int sub) {
        const int nw = threads / 32;
        mw = (P + 31) / 32;
        int o = 0;
        tab = o;     o += TB ? (1 << TB) : 0;
        uv = o;      o += threads * R * 2;
        wt = o;      o += threads * R;
        wfirst = o;  o += threads;
        bars = o;    o += stages;
        tickets = o; o += (stages + 1) / 2 * 2;
        if (o & 1) ++o;
        slot0 = o;
        int q = 0;
        coef = q;    q += spg * P * 8;
        part = q;    q += spg * kPartDoubles;
        far = q;     q += spg * nw * sub * kFarPoly;
        anchor = q;  q += spg * nw * 2;
        mask = q;    q += ((spg * nw * mask_words_per_region(P, sub) + 3) / 4) * 2;
        slot = q;
        total = slot0 + stages * slot;
    }
};
struct F32Smem {
    int uv, wt, bar, wpart, coef, part, far, anchor, mask, coef32, far32, mw, total;
    F32Smem(int sp, int P, int threads, int R) {
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
        coef32 = o; o += sp * P * 4;
        far32 = o;  o += (sp * nw * kFarPoly + 1) / 2;
        o = (o + 1) & ~1;
        total = o;
    }
};
int objective_tiles(int N, const ObjTune& t) { return (N + t.threads * t.r - 1) / (t.threads * t.r); }
size_t objective_smem_bytes(int P, const ObjTune& t, int kk) {
    return (size_t)ObjSmem(t.sp, P, t.threads / 32, t.r, t.tb, kk ? 2 : 1).total * sizeof(double);
}
size_t objective_uniform_smem_bytes(int P, const ObjTune& t, int sub) {
    return (size_t)UniSmem(t.sp, P, t.threads, t.r, t.tb, 2, sub).total * sizeof(double);
}
size_t objective_stream_smem_bytes(int P, const ObjTune& t, int sub) {
    return (size_t)StreamSmem(t.sp, t.stages, P, t.threads, t.r, t.tb, sub).total * sizeof(double);
}
size_t objective_f32_smem_bytes(int P, const ObjTune& t) {
    return (size_t)F32Smem(t.sp, P, t.threads, t.r).total * sizeof(double);
}

// ---- cabi.cu: the context fields these read
struct Ctx {
    int N, P, B, precision, algorithm, far_cells;
    bool uniform;                                          // every spectrum
    ObjTune user_tune;
};
bool use_uniform(const Ctx* c, int fit_im) {
    if (c->algorithm == NMRFIT_ALGO_GENERAL) return false;
    if (fit_im == NMRFIT_IM_SUM || (fit_im == NMRFIT_IM_REFERENCE && c->precision != NMRFIT_FP64)) return false;
    return c->uniform;
}
int ctx_cells(const Ctx* c, int r) { return c->far_cells ? c->far_cells : far_cells_per_region(c->N, r); }
ObjTune pick_tune(const Ctx* c, int S, bool uni) {
    ObjTune t;
    if (uni) {
        if (c->N >= 2048) { t.threads = 256; t.r = 8; }
        else { t.threads = 128; t.r = 4; }
    } else {
        if (c->N >= 8192) { t.threads = 256; t.r = 4; }
        else if (c->N >= 1024) { t.threads = 128; t.r = 4; }
        else { t.threads = 128; t.r = 2; }
    }
    t.tb = 6;
    if (c->user_tune.threads) t.threads = c->user_tune.threads;
    if (c->user_tune.r) t.r = c->user_tune.r;
    if (c->user_tune.tb == -1) t.tb = 0;
    else if (c->user_tune.tb > 0) t.tb = c->user_tune.tb;
    int n_tiles = (c->N + t.threads * t.r - 1) / (t.threads * t.r);
    long long ctas1 = (long long)n_tiles * S * c->B;
    int sp = (int)std::max<long long>(1, std::min<long long>(16, ctas1 / (148 * 4)));
    sp = std::min(sp, std::max(1, S));
    if (c->user_tune.sp > 0) sp = std::min(c->user_tune.sp, std::max(1, S));
    t.sp = sp;
    t.variant = 0;
    t.stages = 0;
    t.occ = 3;
    const long long particle_tiles = (long long)((c->N + t.threads * t.r - 1) / (t.threads * t.r)) * S * c->B;
    const bool enough = particle_tiles >= 8192 || c->user_tune.variant == 1;
    if (uni && c->precision == NMRFIT_FP64 && c->user_tune.variant != 0 && t.tb == 6 && enough) {
        t.variant = 1;
        t.occ = c->user_tune.occ == 3 ? 3 : 2;
        const size_t budget = t.occ == 2 ? 115712 : 74 * 1024;
        const int cells = ctx_cells(c, t.r), per_warp = t.occ == 2 ? cells : 1;
        auto fit_sp = [&](int stg) {
            t.stages = stg;
            int spg = 0;
            for (int cand = 1; cand <= 16; ++cand) {
                t.sp = cand;
                if (objective_stream_smem_bytes(c->P, t, cells) <= budget && (cand < per_warp || cand % per_warp == 0))
                    spg = cand;
            }
            return spg;
        };
        int stg = c->user_tune.stages > 0 ? c->user_tune.stages : 3;
        int spg = fit_sp(stg);
        if (c->user_tune.stages == 0 && spg < 6) {
            const int spg2 = fit_sp(2);
            if (spg2 > spg) { stg = 2; spg = spg2; }
        }
        t.stages = stg;
        t.sp = std::max(1, spg);
        bool fits = true;
        if (c->user_tune.sp > 0) {
            t.sp = c->user_tune.sp;
            if (objective_stream_smem_bytes(c->P, t, ctx_cells(c, t.r)) > 200 * 1024 && c->user_tune.stages == 0) t.stages = 2;
            fits = objective_stream_smem_bytes(c->P, t, ctx_cells(c, t.r)) <= 200 * 1024;
        }
        if (fits) {
            t.sp = std::min(t.sp, std::max(1, S));
            return t;
        }
        t.variant = 0;
        t.stages = 0;
        t.occ = 3;
    }
    const bool f32 = c->precision == NMRFIT_FP32;
    auto uni_bytes = [&]() { return f32 ? objective_f32_smem_bytes(c->P, t) : objective_uniform_smem_bytes(c->P, t, ctx_cells(c, t.r)); };
    while (t.sp > 1 && (uni ? uni_bytes() : objective_smem_bytes(c->P, t, 2)) > 200 * 1024)
        t.sp /= 2;
    if (uni && c->user_tune.sp <= 0)
        while (t.sp > 4 && uni_bytes() > 74 * 1024) t.sp -= 1;
    return t;
}

// launch_objective_prepare: particles and threads per CTA, dynamic shared memory; fills sp / n_tiles / nw
struct Prep { int G, threads; size_t bytes; };
Prep prepare(int N, int P, int S, int B, int sub, const ObjTune& t) {
    const int n_tiles = objective_tiles(N, t), nw = t.threads / 32;
    if (sub < 1) sub = 1;
    const int nc = n_tiles * nw * sub;
    const size_t per_particle = (size_t)(P * 12 + 4 + 3 * P) * sizeof(double);
    int G = std::max(1, std::min(16, std::min(S, 4 * 256 / nc)));
    while (G > 1 && G * per_particle > 40 * 1024) --G;
    int pthreads = nc >= 128 ? 128 : 256;
    if (nc >= 128) G = 1;
    const long long want_ctas = 2 * 148;
    if ((long long)S * B / G < want_ctas) {
        G = (int)std::max<long long>(1, std::min<long long>(G, (long long)S * B / want_ctas));
        if (G == 1) pthreads = 128;
    }
    return {G, pthreads, G * per_particle};
}
int stream_groups_per_cta(int S, int sp, int n_tiles, int B) {
    const long long n_groups = (S + sp - 1) / sp;
    long long gpc = n_groups * n_tiles * B / (148 * 3 * 5);
    gpc = std::max<long long>(4, std::min<long long>(32, gpc));
    const long long chunks = (n_groups + gpc - 1) / gpc;
    return (int)((n_groups + chunks - 1) / chunks);
}

// run_objective past its argument checks, and the launcher it called: the same fields as ObjPlan
nmrfit::ObjPlan run_objective(const Ctx* c, int S, int fit_im, size_t slots_total) {
    nmrfit::ObjPlan p{};
    const bool uni = use_uniform(c, fit_im);
    if (c->algorithm == NMRFIT_ALGO_UNIFORM && !uni) {
        p.refuse = NMRFIT_ERR_STATE;
        p.why = "the uniform-axis kernel needs uniformly spaced w in every spectrum and fit_im off";
        return p;
    }
    if (c->precision == NMRFIT_FP32 && fit_im != NMRFIT_REAL_ONLY) {
        p.refuse = NMRFIT_ERR_ARG;
        p.why = "fit_im is not available in FP32 mode (the Kramers-Kronig term runs in FP64 only)";
        return p;
    }
    ObjTune t = pick_tune(c, S, uni);
    if (uni && c->precision == NMRFIT_FP32 && t.r == 16) t.r = 8;
    if (uni ? (t.r != 4 && t.r != 8 && t.r != 16) : (t.r != 2 && t.r != 4 && t.r != 8)) {
        p.refuse = NMRFIT_ERR_ARG;
        p.why = uni ? "points_per_thread must be 4, 8 or 16 for the uniform-axis kernel"
                    : "points_per_thread must be 2, 4 or 8 for the general kernel";
        return p;
    }
    int n_tiles = objective_tiles(c->N, t);
    p.slots = std::max((size_t)c->B * S, slots_total);
    p.part_per = (size_t)n_tiles * 2 * (t.variant == 1 ? t.threads / 32 : 1);
    const int sub = (uni && c->precision == NMRFIT_FP64) ? ctx_cells(c, t.r) : 1;
    if (uni) {
        const size_t nrp = (size_t)objective_tiles(c->N, t) * (t.threads / 32);
        p.coef = (size_t)c->P * 8;
        p.part = kPartDoubles;
        p.far = nrp * sub * kFarPoly;
        p.anchor = nrp * 2;
        p.mask = nrp * mask_words_per_region(c->P, sub);
        p.pad = kPadParticles;
    }
    p.nsum = c->precision == NMRFIT_FP32 ? 1 : (fit_im ? 2 : 1);
    p.nw = 1;
    p.sub = sub;
    p.t = t;
    if (c->precision == NMRFIT_FP32) {                     // launch_objective_f32
        if (uni) {
            p.kernel = nmrfit::OBJ_F32_UNIFORM;
            p.sub = 1;
            const Prep pr = prepare(c->N, c->P, S, c->B, 1, t);
            p.prep_g = pr.G; p.prep_threads = pr.threads; p.prep_smem = pr.bytes;
            p.n_tiles = objective_tiles(c->N, t);
            p.smem = (size_t)F32Smem(t.sp, c->P, t.threads, t.r).total * sizeof(double);
        } else {
            p.kernel = nmrfit::OBJ_F32_GENERAL;
            p.t.threads = 256; p.t.r = 4;
            p.n_tiles = (c->N + 256 * 4 - 1) / (256 * 4);
            p.smem = ((size_t)t.sp * c->P * 3 + (size_t)t.sp * (256 / 32)) * sizeof(double);
        }
    } else if (uni) {                                      // launch_objective_uniform
        p.tile_major = t.variant == 1;
        const Prep pr = prepare(c->N, c->P, S, c->B, sub, t);
        p.prep_g = pr.G; p.prep_threads = pr.threads; p.prep_smem = pr.bytes;
        p.n_tiles = objective_tiles(c->N, t);
        if (t.variant == 1) {
            p.kernel = nmrfit::OBJ_STREAM;
            p.gpc = stream_groups_per_cta(S, t.sp, p.n_tiles, c->B);
            p.nw = t.threads / 32;
            p.smem = (size_t)StreamSmem(t.sp, t.stages, c->P, t.threads, t.r, t.tb, sub).total * sizeof(double);
        } else {
            p.kernel = nmrfit::OBJ_UNIFORM;
            p.smem = (size_t)UniSmem(t.sp, c->P, t.threads, t.r, t.tb, fit_im ? 2 : 1, sub).total * sizeof(double);
        }
    } else {                                               // launch_objective
        p.kernel = nmrfit::OBJ_GENERAL;
        p.n_tiles = n_tiles;
        p.smem = (size_t)ObjSmem(t.sp, c->P, t.threads / 32, t.r, t.tb, fit_im ? 2 : 1).total * sizeof(double);
    }
    return p;
}
}  // namespace parent

static bool same_tune(const nmrfit::ObjTune& a, const nmrfit::ObjTune& b) {
    return a.threads == b.threads && a.r == b.r && a.tb == b.tb && a.sp == b.sp && a.variant == b.variant &&
           a.stages == b.stages && a.occ == b.occ;
}

// the run fields of two plans (a refused call runs nothing: its refusal alone)
static bool same_run(const nmrfit::ObjPlan& o, const nmrfit::ObjPlan& n) {
    if (o.refuse || n.refuse) return o.refuse == n.refuse && std::strcmp(o.why ? o.why : "", n.why ? n.why : "") == 0;
    return o.kernel == n.kernel && same_tune(o.t, n.t) && o.sub == n.sub && o.n_tiles == n.n_tiles && o.nw == n.nw &&
           o.nsum == n.nsum && o.tile_major == n.tile_major && o.gpc == n.gpc && o.prep_g == n.prep_g &&
           o.prep_threads == n.prep_threads && o.smem == n.smem && o.prep_smem == n.prep_smem && o.slots == n.slots &&
           o.part_per == n.part_per && o.coef == n.coef && o.part == n.part && o.far == n.far && o.anchor == n.anchor &&
           o.mask == n.mask && o.pad == n.pad;
}

int main() {
    const int Ns[] = {1, 2, 31, 257, 1000, 1024, 2047, 2048, 4096, 8191, 8192, 16384, 32768, 65536, 2100000};
    const int Ps[] = {1, 6, 12, 24, 64}, Ss[] = {1, 100, 204, 4096, 65536}, Bs[] = {1, 24, 1024};
    const int threads_v[] = {0, 128, 256}, r_v[] = {0, 2, 4, 8, 16}, tb_v[] = {0, -1, 6, 8, 10};
    const int sp_v[] = {SP_VALUES};
    const int variant_v[] = {-1, 0, 1}, stages_v[] = {0, 2, 3, 4}, occ_v[] = {0, 2, 3}, far_v[] = {0, 1, 2, 4};
    const int n_shape = 15 * 5 * 5 * 3;
    std::atomic<long long> cases{0}, run_cases{0}, refused{0}, run_diff{0}, algo_diff{0}, variant_diff{0};
    std::atomic<long long> tuning_same{0}, tuning_f32_r16{0}, tuning_f32_general{0}, tuning_other{0};
    std::atomic<long long> by_kernel[5] = {};
#pragma omp parallel for schedule(dynamic)
    for (int shape = 0; shape < n_shape; ++shape) {
        const int N = Ns[shape % 15], P = Ps[shape / 15 % 5], S = Ss[shape / 75 % 5], B = Bs[shape / 375];
        long long n_cases = 0, n_run = 0, n_ref = 0, d_run = 0, d_algo = 0, d_var = 0, t_same = 0, t_r16 = 0, t_gen = 0,
                  t_other = 0, kern[5] = {};
        for (int prec : {NMRFIT_FP64, NMRFIT_FP32})
        for (int uniform : {0, 1})
        for (int algo : {NMRFIT_ALGO_AUTO, NMRFIT_ALGO_GENERAL, NMRFIT_ALGO_UNIFORM})
        for (int th : threads_v) for (int r : r_v) for (int tb : tb_v)
        for (int sp : sp_v)
        for (int var : variant_v) for (int stg : stages_v) for (int occ : occ_v) for (int far : far_v) {
            const nmrfit::ObjTune user{th, r, tb, sp, var, stg, occ};
            const parent::Ctx c{N, P, B, prec, algo, far, uniform != 0, user};
            // nmrfit_ctx_get_tuning / _get_variant: the real-only plan, refused or not
            const nmrfit::ObjTune ot = parent::pick_tune(&c, S, parent::use_uniform(&c, NMRFIT_REAL_ONLY));
            const nmrfit::ObjPlan q = nmrfit::objective_plan(N, P, S, B, prec, NMRFIT_REAL_ONLY, uniform, algo, user, far);
            if (ot.variant != q.t.variant || ot.stages != q.t.stages) ++d_var;
            const bool rep_same = ot.threads == q.t.threads && ot.r == q.t.r && ot.tb == q.t.tb && ot.sp == q.t.sp &&
                                  parent::objective_tiles(N, ot) == q.n_tiles;
            if (rep_same) ++t_same;
            else if (prec == NMRFIT_FP32 && q.kernel == nmrfit::OBJ_F32_UNIFORM && ot.r == 16 && q.t.r == 8 &&
                     ot.threads == q.t.threads && ot.tb == q.t.tb && ot.sp == q.t.sp)
                ++t_r16;
            else if (prec == NMRFIT_FP32 && q.kernel == nmrfit::OBJ_F32_GENERAL && q.t.threads == 256 && q.t.r == 4 &&
                     q.n_tiles == (N + 1023) / 1024 && ot.tb == q.t.tb && ot.sp == q.t.sp)
                ++t_gen;
            else
                ++t_other;
            for (int fit_im = 0; fit_im <= 2; ++fit_im)
            for (size_t slots_total : {(size_t)0, (size_t)300000}) {
                ++n_cases;
                const nmrfit::ObjPlan o = parent::run_objective(&c, S, fit_im, slots_total);
                const nmrfit::ObjPlan n = nmrfit::objective_plan(N, P, S, B, prec, fit_im, uniform, algo, user, far,
                                                                 slots_total);
                if (o.refuse) ++n_ref;
                else { ++n_run; ++kern[o.kernel]; }
                if (!same_run(o, n)) ++d_run;
                const bool ou = parent::use_uniform(&c, fit_im);
                const bool nu = n.kernel != nmrfit::OBJ_GENERAL && n.kernel != nmrfit::OBJ_F32_GENERAL;
                if (ou != nu) ++d_algo;
            }
        }
        cases += n_cases; run_cases += n_run; refused += n_ref; run_diff += d_run; algo_diff += d_algo;
        variant_diff += d_var; tuning_same += t_same; tuning_f32_r16 += t_r16; tuning_f32_general += t_gen;
        tuning_other += t_other;
        for (int k = 0; k < 5; ++k) by_kernel[k] += kern[k];
    }
    std::printf("objective_plan against the parent's pick_tune, run_objective and launchers\n");
    std::printf("grid: N %d values x P 5 x S 5 x B 3 x precision 2 x uniform axis 2 x algorithm 3 x threads 3 x r 5 x "
                "tb 5 x sp %s x variant 3 x stages 4 x occupancy 3 x far cells 4\n", 15, SP_NAME);
    std::printf("calls (x fit_im 0/1/2 x sliced or not): %lld; run %lld, refused %lld\n", cases.load(), run_cases.load(),
                refused.load());
    const char* names[5] = {"general FP64", "uniform one-group", "uniform streamed", "FP32 uniform", "FP32 general"};
    for (int k = 0; k < 5; ++k) std::printf("  runs on %-18s %lld\n", names[k], by_kernel[k].load());
    std::printf("calls whose plan differs (kernel, geometry, smem, scratch, refusal): %lld\n", run_diff.load());
    std::printf("get_algorithm differs: %lld\n", algo_diff.load());
    std::printf("get_variant differs: %lld\n", variant_diff.load());
    std::printf("get_tuning: same %lld; FP32 uniform asked r = 16, now reports the r = 8 that runs: %lld; FP32 on a "
                "non-uniform axis, now reports the 256 x 4 and tile count that run: %lld; any other difference: %lld\n",
                tuning_same.load(), tuning_f32_r16.load(), tuning_f32_general.load(), tuning_other.load());
    const bool ok = run_diff == 0 && algo_diff == 0 && variant_diff == 0 && tuning_other == 0;
    std::printf("%s\n", ok ? "EQUIVALENT (up to the two reporting changes)" : "DIFFERENT");
    return ok ? 0 : 1;
}
