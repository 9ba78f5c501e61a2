// The two device routines of the uniform-axis objective, shared by the two-pass kernels
// (objective_uniform.cu, objective_stream.cu) and the fused swarm kernel (swarm_fused.cu) so that all of them
// evaluate a particle with the SAME arithmetic in the SAME order - their objective values are bit-identical.
//
//   prepare_particle  per-particle constants: span coefficients of its peaks, phase tables and, per
//                     far-field CELL, the near-peak mask and the far-field polynomial; per region of 32*R points
//                     the phase anchor.  The destinations are plain pointers: global memory in the
//                     two-pass path, shared memory in the fused kernel.
//   eval_region       one warp's squared weighted residual over its region, from those constants
//                     and the staged (u, v, weights) of the tile.
//   eval_region_multi the same sum for `sub` particles at once, one per group of 32/sub lanes, cell by cell
//                     (the streamed kernel); both are made of the same per-lane steps.
//
// Regions and cells.  A warp evaluates a REGION of 32*R consecutive points (a thread R of them).  The far-field
// polynomial (nmrfit_math.cuh) lives on a CELL: the region itself, or one half / quarter of it (`sub` = 1, 2, 4 cells
// per region, i.e. 32 / sub lanes each).  A peak is far from a cell when its centre is >= 8 cell lengths away (and
// its Gaussian cannot reach the cell), so shorter cells leave fewer peaks to evaluate one by one: on a 4,096-point
// axis with 6 peaks, 4.75 of them are near the average 256-point region but only 1.6 near the average 64-point cell.
// The price is `sub` times the polynomials in the prepare pass, so long axes (where the Gaussian's reach, not the
// series, decides what is near) keep sub = 1: far_cells_per_region() in nmrfit_internal.h, a function of the axis
// length and R alone - never of how particles or spectra are sharded.
#pragma once
#include <cuda_runtime.h>
#include "nmrfit_math.cuh"
#include "uniform_common.cuh"

namespace nmrfit {

// 32-bit mask words per region: one cell - [MW near words][has-far]; several cells - the same block for the UNION of
// the region's cells first (what the warp as a whole has to visit), then one block per cell.
__host__ __device__ inline int mask_words_per_region(int P, int sub) { return (sub == 1 ? 1 : sub + 1) * ((P + 31) / 32 + 1); }

// ---- the items of the prepare pass.  One particle's constants are a few dozen independent work items; the prepare
// kernel (objective_uniform.cu) spreads the items of SEVERAL particles over the threads of a CTA so that no warp idles,
// the fused swarm kernel (one CTA per particle) those of one.  Same item, same arithmetic, whoever executes it.
constexpr int kPairDoubles = kFarTerms + 1;                // a (cell, peak) series: kind, then v[n]
constexpr int kTableItems = 33;                            // phase table: 32 lane factors, the per-point step

// span coefficients of peak k -> cs[k][8] (shared) and optionally a second copy
// (farpk [P][4], shared: what the far-field classification of this peak needs besides the cell's position - A = H dT,
// A^2, 256 A^2 and the Gaussian's reach for cells of 32 R / sub points, nmrfit_math.cuh make_far_peak)
template <int R>
__device__ __forceinline__ void prep_item_coef(const double* __restrict__ xs, int k, double h, double w_ulp,
                                               double* __restrict__ cs, double* __restrict__ coef_out,
                                               double* __restrict__ farpk, int sub, int P, double* __restrict__ part) {
    if (k == 0) part[66] = (double)P * xs[3];              // yoff is added once per peak (equations.py:147,195)
    SpanCoef c = make_span_coef(xs[2], xs[4 + 3 * k], xs[5 + 3 * k], xs[6 + 3 * k], h, w_ulp, R);
    if (c.exact) c = null_span_coef();                     // the span loop adds zero; the peak is handled after it
    double* o = cs + k * 8;
    o[0] = c.loc; o[1] = c.kL; o[2] = c.kG; o[3] = c.aL; o[4] = c.aG; o[5] = c.dT; o[6] = c.thr; o[7] = c.c2;
    const FarPeak f = make_far_peak(c, 0.5 * (double)(32 * R / sub));
    double* q = farpk + k * 4;
    q[0] = f.A; q[1] = f.A2; q[2] = f.A2x; q[3] = f.reach;
    if (coef_out) {
        double* g = coef_out + k * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) g[i] = o[i];
    }
}

// The rotation items of a particle - kTableItems entries of its phase table, then one anchor per region - are all "one
// angle -> (cos, sin)": item `it` of a particle yields its angle here and the caller takes ONE sincos for whatever
// mix of items its warp holds (they used to be two call sites: a warp with both paid for both).
//   phi_i = p0 + (p1*i)/N with i = i_r + lane*R + j is anchor(i_r) * e^{i p1 (lane R)/N} * (e^{i p1/N})^j:
//   items 0..31 the lanes' factors, 32 the per-point step (-> part[2*it]), 33 + ra the phase at the first point of
//   region ra (-> the region's anchor; regions past the end of the axis get angle 0: cos 1, sin 0).
// (inv_N = 1.0 / N, taken once per thread: a division per item cost ~25 instructions, and the items whose numerator
// is zero - lane 0, region 0 - sent their whole warp through the division's slow path on top.)
template <int R>
__device__ __forceinline__ double prep_item_angle(const double* __restrict__ xs, int it, int N, double inv_N) {
    if (it < 32) return (xs[1] * (double)(it * R)) * inv_N;
    if (it == 32) return xs[1] * inv_N;
    const int ra = it - kTableItems;
    return (long long)ra * 32 * R < N ? fma(xs[1] * (double)(ra * 32 * R), inv_N, xs[0]) : 0.0;
}

// e / d for 0 <= e < 2^22 with inv = 1.0f / d (exact after one correction step): the prepare pass maps flat item
// numbers to (particle, item) a few times per thread, and an integer division is ~20 instructions
__device__ __forceinline__ int fast_div(int e, int d, float inv) {
    int q = __float2int_rz(__int2float_rn(e) * inv);
    const int r = e - q * d;
    q += (r >= d) - (r < 0);
    return q;
}

// number of exact-path peaks (thr < 0 marks a nulled peak) -> part[67]; needs the particle's cs complete
__device__ __forceinline__ void prep_item_exact_count(const double* __restrict__ cs, int P, double* __restrict__ part) {
    int n = 0;
    for (int k = 0; k < P; ++k) n += cs[k * 8 + 6] < 0.0;
    part[67] = (double)n;
}

// the series of one (cell, peak) pair -> pr[kPairDoubles]; `ic` = the cell's first point; needs cs complete
template <int R>
__device__ __forceinline__ void prep_item_pair(const double* __restrict__ cs, const double* __restrict__ farpk,
                                               const double* __restrict__ sw, double h, int N,
                                               int sub, long long ic, int k, double* __restrict__ pr) {
    const int cell_pts = 32 * R / sub;
    double kind = -1.0;                                    // -1: padding cell or exact-path peak (neither near nor far)
    if (ic < N) {
        const double* o = cs + k * 8;
        if (!(o[6] < 0.0)) {
            const double* q = farpk + k * 4;
            FarPeak f;
            f.A = q[0]; f.A2 = q[1]; f.A2x = q[2]; f.reach = q[3];
            const double w_c = fma(0.5 * (double)(cell_pts - 1), h, sw[ic]);
            double v[kFarTerms];
            kind = (double)far_terms_pre(w_c - o[0], o[1], o[2], f, v);
#pragma unroll
            for (int n = 0; n < kFarTerms; ++n) pr[1 + n] = v[n];
        }
    }
    pr[0] = kind;
}

// One far-field cell: classify every peak as near / far, sum the far ones' series into the cell's polynomial (peaks in
// index order), write the polynomial and the cell's mask block.  `ic` = the cell's first point (cells past the end of
// the axis are neutral); `pairs_row` (optional): the cell's (cell, peak) series precomputed by prep_item_pair.  Must be
// called by ALL lanes of a warp (`ok` false for lanes without a cell): the union block of a region is combined from
// its `sub` cells - consecutive lanes - by shuffles; mask_region points at the region's first block, ci = cell in region.
template <int R>
__device__ __forceinline__ void prep_item_cell(bool ok, const double* __restrict__ cs, const double* __restrict__ farpk,
                                               const double* __restrict__ sw, double h, int N, int P, int sub, long long ic, int ci,
                                               const double* __restrict__ pairs_row, double* __restrict__ far_dst,
                                               unsigned* __restrict__ mask_region) {
    const int MW = (P + 31) / 32;
    const int cell_pts = 32 * R / sub;
    double C[kFarTerms];
#pragma unroll
    for (int n = 0; n < kFarTerms; ++n) C[n] = 0.0;
    unsigned any_far = 0;
    unsigned* mk = mask_region + (sub == 1 ? 0 : 1 + ci) * (MW + 1);
    const bool live = ok && ic < N;
    const double w_c = (live && !pairs_row) ? fma(0.5 * (double)(cell_pts - 1), h, sw[ic]) : 0.0;
    for (int wd = 0; wd < MW; ++wd) {
        unsigned m = 0;
        if (live) {
            const int kend = min(P, wd * 32 + 32);
            for (int k = wd * 32; k < kend; ++k) {
                if (pairs_row) {
                    const double* pr = pairs_row + (size_t)k * kPairDoubles;
                    const int kind = (int)pr[0];
                    if (kind < 0) continue;
                    if (kind == kFarNear) { m |= 1u << (k & 31); continue; }
                    any_far = 1u;
                    if (kind == kFarSeries) {
                        double v[kFarTerms];
#pragma unroll
                        for (int n = 0; n < kFarTerms; ++n) v[n] = pr[1 + n];
                        far_add(cs[k * 8 + 3], v, C);
                    }
                } else {
                    const double* o = cs + k * 8;
                    if (o[6] < 0.0) continue;              // exact-path peak (thr < 0): neither near nor far
                    const double2 c01 = *reinterpret_cast<const double2*>(o);            // loc, kL
                    const double2 c23 = *reinterpret_cast<const double2*>(o + 2);        // kG, aL
                    const double2 f01 = *reinterpret_cast<const double2*>(farpk + k * 4);
                    const double2 f23 = *reinterpret_cast<const double2*>(farpk + k * 4 + 2);
                    FarPeak f;
                    f.A = f01.x; f.A2 = f01.y; f.A2x = f23.x; f.reach = f23.y;
                    double v[kFarTerms];
                    const int kind = far_terms_pre(w_c - c01.x, c01.y, c23.x, f, v);
                    if (kind == kFarNear) { m |= 1u << (k & 31); continue; }
                    any_far = 1u;
                    if (kind == kFarSeries) far_add(c23.y, v, C);
                }
            }
        }
        if (ok) mk[wd] = m;
        if (sub > 1) {                                     // the region's union: its cells sit in `sub` consecutive lanes
            unsigned mu = m;
            for (int o = 1; o < sub; o <<= 1) mu |= __shfl_xor_sync(0xffffffffu, mu, o);
            if (ok && ci == 0) mask_region[wd] = mu;
        }
    }
    if (ok) mk[MW] = any_far;
    if (sub > 1) {
        unsigned fu = any_far;
        for (int o = 1; o < sub; o <<= 1) fu |= __shfl_xor_sync(0xffffffffu, fu, o);
        if (ok && ci == 0) mask_region[MW] = fu;
    }
    if (ok) {
        far_economise(C);                                  // 12 series terms -> kFarPoly stored coefficients
#pragma unroll
        for (int n = 0; n < kFarPoly; n += 2) *reinterpret_cast<double2*>(far_dst + n) = make_double2(C[n], C[n + 1]);
    }
}

// All items of ONE particle by the `nthreads` (a multiple of 32) threads of a CTA - what the fused swarm kernel runs
// per generation.  xs: the particle's D parameters; sw: its spectrum's w plane (N points); cs: shared [P][8] scratch
// that ends up holding the span coefficients; farpk: shared [P][4] scratch (per-peak far-field constants);
// coef_out: optional second copy of the coefficients; part [kPartDoubles];
// far [cells][kFarPoly]; anchor [regions][2]; mask [regions][mask_words_per_region].  Regions [r_lo, r_hi) are filled,
// at index r - r_lo (default: all NRP slots; the slots of regions past the end of the axis are neutral).  Contains
// __syncthreads().  `pairs` (optional shared scratch of cells*P*kPairDoubles doubles): the (cell, peak) series are
// computed one pair per thread instead of one cell per thread - same values, same order of accumulation, but P times
// shorter on the critical path.
template <int R>
__device__ __forceinline__ void prepare_particle(const double* __restrict__ xs, const double* __restrict__ sw, double h,
                                                 double w_ulp, int N, int P, int NR, int NRP, int tid, int nthreads,
                                                 double* __restrict__ cs, double* __restrict__ coef_out,
                                                 double* __restrict__ part, double* __restrict__ far,
                                                 double* __restrict__ anchor, unsigned* __restrict__ mask,
                                                 double* __restrict__ farpk, double* __restrict__ pairs = nullptr,
                                                 int r_lo = 0, int r_hi = -1, int sub = 1) {
    if (r_hi < 0) r_hi = NRP;
    const int nr = r_hi - r_lo, nc = nr * sub;
    const int cell_pts = 32 * R / sub;
    const int MWR = mask_words_per_region(P, sub);
    (void)NR;
    for (int k = tid; k < P; k += nthreads) prep_item_coef<R>(xs, k, h, w_ulp, cs, coef_out, farpk, sub, P, part);
    // the threads at the far end of the CTA do the phase table and the anchors while the first do the peaks
    const double inv_N = 1.0 / (double)N;
    for (int e = nthreads - 1 - tid; e < kTableItems + nr; e += nthreads) {
        double sn, cn;
        sincos(prep_item_angle<R>(xs, e < kTableItems ? e : e + r_lo, N, inv_N), &sn, &cn);
        double* dst = e < kTableItems ? part + 2 * e : anchor + 2 * (e - kTableItems);
        dst[0] = cn;
        dst[1] = sn;
    }
    __syncthreads();
    if (tid == nthreads - 1) prep_item_exact_count(cs, P, part);
    if (pairs) {
        for (int pi = tid; pi < nc * P; pi += nthreads) {  // one (cell, peak) pair per thread, in rounds
            const int cl = pi / P, k = pi - cl * P;
            prep_item_pair<R>(cs, farpk, sw, h, N, sub, ((long long)r_lo * sub + cl) * cell_pts, k,
                              pairs + (size_t)pi * kPairDoubles);
        }
        __syncthreads();
    }
    for (int base = tid & ~31; base < nc; base += nthreads) {      // whole warps: prep_item_cell shuffles
        const int cl = base + (tid & 31);
        const bool ok = cl < nc;
        const int rl = cl / sub, ci = cl - rl * sub;
        prep_item_cell<R>(ok, cs, farpk, sw, h, N, P, sub, ((long long)r_lo * sub + cl) * cell_pts, ci,
                          pairs ? pairs + (size_t)cl * P * kPairDoubles : nullptr, far + (size_t)cl * kFarPoly,
                          mask + (size_t)rl * MWR);
    }
}

// Shared-memory placement of a tile's staged points.  Point e of the tile (thread t = e / R, j = e % R) lives in
// row j.  Swizzled (SWZ): at column t ^ j (double2 (u, v) array) resp. t ^ 2j (weights array) - the evaluation reads
// row j with consecutive t (a permutation inside each aligned group of 16 columns: conflict-free), and the staging
// loop, whose consecutive lanes hold consecutive e - eight different rows of the same column - spreads over eight
// different banks instead of colliding 8-way.  Plain (!SWZ): at column t; the staging stores collide, which a kernel
// that stages once per CTA and then evaluates hundreds of particles (objective_stream.cu) does not notice, and the
// evaluation's addresses are one base plus compile-time offsets - no integer work per point.
// What the evaluation kernels stage per point: the data pre-multiplied by the residual weights - the residual
// weights * (u cos - v sin - V_fit) then costs one multiply less per (particle, point).
__device__ __forceinline__ double2 stage_point(double u, double v, double wt) {
    return make_double2(__dmul_rn(wt, u), __dmul_rn(wt, v));
}
__device__ __forceinline__ int stage_slot_uv(int t, int j, int stride) { return j * stride + (t ^ j); }
__device__ __forceinline__ int stage_slot_wt(int t, int j, int stride) { return j * stride + (t ^ (2 * j)); }

// Where a lane's far-field cell keeps its mask block and its polynomial inside the region's constants: loop-invariant,
// computed once per thread (mk_off == 0 <=> the region is one cell and has no separate union block).
struct LaneCell { int mk_off, fc_off, mirror; };       // mirror: xor mask to the lane holding the mirror-image span
__device__ __forceinline__ LaneCell lane_cell(int lane, int sub, int P) {
    const int cell = (lane * sub) >> 5, MW = (P + 31) / 32;
    LaneCell lc;
    lc.mk_off = sub == 1 ? 0 : (1 + cell) * (MW + 1);
    lc.fc_off = cell * kFarPoly;
    lc.mirror = 32 / sub - 1;
    return lc;
}

// The per-lane steps of a region's evaluation, shared by eval_region and eval_region_multi so that a point gets the
// same arithmetic in the same order whichever of them evaluates it.
//
// Far field: the cell's polynomial fcc [kFarPoly] (plus P*yoff) at the lane's R points - all far peaks of the cell at
// once.  A cell without far peaks holds zeros: evaluated all the same - rare, and a branch here costs every other cell a
// dozen instructions.  The last R/2 points are the mirror image, inside the cell, of the first R/2 points of lane ^ mirror.
template <int R>
__device__ __forceinline__ void lane_far_start(const double* __restrict__ fcc, double py, double xi0, double inv_H,
                                               int mirror, double (&acc)[R]) {
    double C[kFarPoly];
#pragma unroll
    for (int n = 0; n < kFarPoly; n += 2) {
        const double2 t2 = *reinterpret_cast<const double2*>(fcc + n);
        C[n] = t2.x; C[n + 1] = t2.y;
    }
    C[0] += py;
    double mir[R / 2];
    far_init_half<R>(C, xi0, inv_H, acc, mir);
#pragma unroll
    for (int j = 0; j < R / 2; ++j) acc[R - 1 - j] = __shfl_xor_sync(0xffffffffu, mir[j], mirror);
}

// near peak k (span coefficients cf [P][8]) at the lane's R points
template <int R, int TB>
__device__ __forceinline__ void lane_near_peak(const double* __restrict__ cf, int k, double w_first,
                                               const double* __restrict__ tab, double (&acc)[R]) {
    const double2 c01 = *reinterpret_cast<const double2*>(cf + k * 8);
    const double2 c23 = *reinterpret_cast<const double2*>(cf + k * 8 + 2);
    const double2 c45 = *reinterpret_cast<const double2*>(cf + k * 8 + 4);
    const double2 c67 = *reinterpret_cast<const double2*>(cf + k * 8 + 6);
    SpanCoef c;
    c.loc = c01.x; c.kL = c01.y; c.kG = c23.x; c.aL = c23.y;
    c.aG = c45.x; c.dT = c45.y; c.thr = c67.x; c.c2 = c67.y;
    peak_span<R, TB>(w_first - c.loc, c, tab, acc);
}

// rare: peaks too narrow for the uniform-axis shortcuts, from the particle's parameters xs and the stored abscissae
template <int R, int TB>
__device__ __forceinline__ void lane_exact_peaks(const double* __restrict__ cf, const double* __restrict__ pt, int P,
                                                 const double* __restrict__ xs, const double* __restrict__ sw_first,
                                                 int n_valid, double w_first, double h, double w_ulp,
                                                 const double* __restrict__ tab, double (&acc)[R]) {
    if (pt[67] != 0.0) {
        for (int k = 0; k < P; ++k) {
            if (!(cf[k * 8 + 6] < 0.0)) continue;
            const SpanCoef c = make_span_coef(xs[2], xs[4 + 3 * k], xs[5 + 3 * k], xs[6 + 3 * k], h, w_ulp, R);
            peak_exact<R, TB>(sw_first, n_valid, w_first, h, c, tab, acc);
        }
    }
}

// the lane's sum of squared weighted residuals against the phase-rotated data: ew = the region's phase anchor, lf = the
// lane factor's index in the phase table (the lane's thread span inside the region); the rotation advances by p1/N per
// point.  KK also returns the imaginary parts' sum through *ssi.
template <int R, int KK, bool SWZ>
__device__ __forceinline__ double lane_residual(const double (&acc)[R], const double* __restrict__ cf,
                                                const double* __restrict__ pt, int P, const double2 ew, int lf,
                                                const double2* __restrict__ suv, const double* __restrict__ swt, int t,
                                                int stride, const double* __restrict__ xs,
                                                const double* __restrict__ sw_first, int n_valid, double w_first,
                                                double h, double w_ulp, double* ssi_out) {
    const double2 el = *reinterpret_cast<const double2*>(pt + 2 * lf);
    const double cd = pt[64], sd = pt[65];
    double cr = fma(ew.x, el.x, -(ew.y * el.y));
    double ci = fma(ew.y, el.x, ew.x * el.y);
    double ss = 0.0, ssi = 0.0;
    // fit_im is True: I_fit is OVERWRITTEN peak by peak (equations.py:198-199), so only the LAST peak's Kramers-Kronig
    // curve is ever compared with the data.  Its constants are its span coefficients - rebuilt from the parameters
    // when the peak is on the exact path (the shared copy is nulled then).
    double kloc = 0.0, kkL = 0.0, kkG = 0.0, kaL = 0.0, kaG = 0.0;
    bool kexact = false;
    if (KK) {
        const double* cl = cf + (P - 1) * 8;
        kexact = cl[6] < 0.0;
        if (kexact) {
            const int k = P - 1;
            const SpanCoef c = make_span_coef(xs[2], xs[4 + 3 * k], xs[5 + 3 * k], xs[6 + 3 * k], h, w_ulp, R);
            kloc = c.loc; kkL = c.kL; kkG = c.kG; kaL = c.aL; kaG = c.aG * kTwoOverSqrtPi;
        } else {
            kloc = cl[0]; kkL = cl[1]; kkG = cl[2]; kaL = cl[3]; kaG = cl[4] * kTwoOverSqrtPi;
        }
    }
    const double2* puv = suv + t;                          // !SWZ: row j of this thread at a compile-time offset
    const double* pwt = swt + t;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const double2 uv = SWZ ? suv[stage_slot_uv(t, j, stride)] : puv[j * stride];
        const double wt = SWZ ? swt[stage_slot_wt(t, j, stride)] : pwt[j * stride];
        // weights * (V_data - V_fit); the staged data carry the weights: uv = weights * (u, v) (stage_point)
        const double res = fma(uv.x, cr, -fma(uv.y, ci, wt * acc[j]));
        ss = fma(res, res, ss);
        if (KK) {
            const double idat = fma(uv.x, ci, uv.y * cr);  // weights * I_data
            // abscissa: w_first + j*h on the uniform axis; the stored value when the peak is too narrow for that
            const double wj = (kexact && j < n_valid) ? sw_first[j] : (j == 0 ? w_first : fma((double)j, h, w_first));
            const double d = wj - kloc;
            const double tt = d * kkL;
            const double rq = rcp_pos(fma(tt, tt, 1.0));
            const double daw = dawson(d * kkG, NMRFIT_DAW_TAB, NMRFIT_DAW_TAIL);
            const double ifit = fma(kaL * tt, rq, kaG * daw);
            const double ri = fma(-wt, ifit, idat);
            ssi = fma(ri, ri, ssi);
        }
        if (j + 1 < R) {
            const double c2 = fma(cr, cd, -(ci * sd));
            ci = fma(ci, cd, cr * sd);
            cr = c2;
        }
    }
    if (KK) *ssi_out = ssi;
    return ss;
}

// One warp, one particle, one region: sum over the warp's 32*R points of (weights * (V_data - V_fit))^2, identical
// in every lane on return.  cf [P][8], pt [kPartDoubles], mk [mask_words_per_region], fc [sub][kFarPoly] (16-byte aligned) and ew
// are the particle's constants for this region (`sub` far-field cells of 32/sub lanes each, lc = lane_cell(lane, sub, P); xi0 is the lane's first
// point's position inside ITS cell and inv_H the step of that coordinate per point); the R points of thread t of the
// tile sit at stage_slot_uv/wt(t, j, stride) of suv / swt (SWZ) or at j*stride + t (!SWZ); w_first is the abscissa of its
// first point.  The exact path (peaks too narrow for the recurrences) reads the particle's parameters xs and the stored
// abscissae sw_first[0..n_valid).
// SUBT: the number of cells when the caller knows it at compile time (0: take everything from lc).
// KK = 1 (fit_im, reference semantics) also returns through *ss_im the same sum for the imaginary parts:
// I_data = u sin(phi) + v cos(phi) against the last peak's Kramers-Kronig counterpart (closed form, nmrfit_math.cuh).
template <int R, int TB, int KK = 0, bool SWZ = true, int SUBT = 0>
__device__ __forceinline__ double eval_region(const double* __restrict__ cf, const double* __restrict__ pt,
                                              const unsigned* __restrict__ mk, const double* __restrict__ fc,
                                              const double2 ew, int MW, int P, int lane, const LaneCell lc, double w_first, double xi0,
                                              double inv_H, const double2* __restrict__ suv, const double* __restrict__ swt,
                                              int t, int stride, const double* __restrict__ tab,
                                              const double* __restrict__ xs, const double* __restrict__ sw_first,
                                              int n_valid, double h, double w_ulp, double* ss_im = nullptr) {
    const unsigned* mkc = mk + lc.mk_off;                  // this lane's cell; mk itself: the union's block (prepare_particle)
    double acc[R];
    // (P*yoff: yoff is added once per peak, equations.py:147,195)
    lane_far_start<R>(fc + lc.fc_off, pt[66], xi0, inv_H, SUBT ? 32 / SUBT - 1 : lc.mirror, acc);
    for (int wd = 0; wd < MW; ++wd) {
        const unsigned mine = mkc[wd];                     // peaks near this lane's cell
        for (unsigned m = mk[wd]; m; m &= m - 1) {         // peaks near ANY cell of the region (uniform across the warp)
            const int kb = __ffs(m) - 1;
            // (in a cell for which the peak is far it is already inside that cell's polynomial)
            if ((SUBT ? SUBT == 1 : lc.mk_off == 0) || ((mine >> kb) & 1u)) lane_near_peak<R, TB>(cf, wd * 32 + kb, w_first, tab, acc);
        }
    }
    lane_exact_peaks<R, TB>(cf, pt, P, xs, sw_first, n_valid, w_first, h, w_ulp, tab, acc);
    double ssi = 0.0;
    double ss = lane_residual<R, KK, SWZ>(acc, cf, pt, P, ew, lane, suv, swt, t, stride, xs, sw_first, n_valid, w_first,
                                          h, w_ulp, &ssi);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (KK) ssi += __shfl_xor_sync(0xffffffffu, ssi, o);
    }
    if (KK) *ss_im = ssi;
    return ss;
}

// One warp, SUB (2 or 4) particles, one region of SUB far-field cells, real part only: the warp's 32 / SUB-lane group q
// holds particle q and walks the region's cells one pass at a time.  In pass c lane i of a group evaluates the points
// that lane c * 32/SUB + i evaluates in eval_region - same constants, same arithmetic, same order - so every group
// visits only the peaks near cell c of SOME particle of the warp (near sets of particles in one cell hardly differ,
// while the cells of one region often differ by a peak), the staged points are read once for SUB particles, and the
// warp's reduction tree is paid once for SUB particles.  The lane's per-pass sums are added in eval_region's tree:
// its shuffle levels 16 (and 8) pair the passes ((s0 + s2) + (s1 + s3), resp. s0 + s1), then xor 32/SUB/2 .. 1.
// Arguments are the lane's particle's, as for eval_region, except: mk = its region's mask words (the union block
// first), fc = its region's SUB polynomials; t0 = the region's first thread span of the tile, swf = the tile's stored
// first abscissae per thread span, sw_tile = the w plane from the tile's first point on, n_tile = the axis' points from
// there on.  Returns the particle's region sum in every lane of its group; the staged points sit at j*stride + t.
template <int R, int TB, int SUB>
__device__ __forceinline__ double eval_region_multi(const double* __restrict__ cf, const double* __restrict__ pt,
                                                    const unsigned* __restrict__ mk, const double* __restrict__ fc,
                                                    const double2 ew, int MW, int P, int lane, double xi0, double inv_H,
                                                    const double2* __restrict__ suv, const double* __restrict__ swt,
                                                    const double* __restrict__ swf, int t0, int stride,
                                                    const double* __restrict__ tab, const double* __restrict__ xs,
                                                    const double* __restrict__ sw_tile, int n_tile, double h, double w_ulp) {
    static_assert(SUB == 2 || SUB == 4, "one pass per far-field cell of the region");
    constexpr int LPC = 32 / SUB;                          // lanes per cell = lanes per particle
    const int i = lane & (LPC - 1);
    const double py = pt[66];
    double se = 0.0, so = 0.0;                             // sums of the even / odd passes
#pragma unroll 1
    for (int c = 0; c < SUB; ++c) {
        const int lf = c * LPC + i, t = t0 + lf;
        const double w_first = swf[t];
        double acc[R];
        lane_far_start<R>(fc + c * kFarPoly, py, xi0, inv_H, LPC - 1, acc);
        const unsigned* mkc = mk + (1 + c) * (MW + 1);
        for (int wd = 0; wd < MW; ++wd) {
            const unsigned mine = mkc[wd];                 // peaks near cell c of this lane's particle
            for (unsigned m = __reduce_or_sync(0xffffffffu, mine); m; m &= m - 1) {   // ... of any particle of the warp
                const int kb = __ffs(m) - 1;
                if ((mine >> kb) & 1u) lane_near_peak<R, TB>(cf, wd * 32 + kb, w_first, tab, acc);
            }
        }
        lane_exact_peaks<R, TB>(cf, pt, P, xs, sw_tile + t * R, n_tile - t * R, w_first, h, w_ulp, tab, acc);
        const double s = lane_residual<R, 0, false>(acc, cf, pt, P, ew, lf, suv, swt, t, stride, xs, sw_tile + t * R,
                                                    n_tile - t * R, w_first, h, w_ulp, nullptr);
        // (s >= +0: a sum of squares from +0, so 0 + s == s)
        if (c & 1) so += s;
        else se += s;
    }
    double ss = se + so;
#pragma unroll
    for (int o = LPC / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    return ss;
}

// first point's position of a lane inside its far-field cell, in half-cells: xi in (-1, 1)
template <int R>
__device__ __forceinline__ double cell_xi0(int lane, int sub) {
    const int lpc = 32 / sub;                              // lanes per cell
    const double H = 0.5 * (double)(lpc * R);
    return ((double)((lane % lpc) * R) - 0.5 * (double)(lpc * R - 1)) / H;
}

}  // namespace nmrfit
