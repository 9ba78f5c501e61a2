// Internal declarations shared by the translation units of libnmrfit_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <type_traits>
#include "objective_plan.h"

#define NMRFIT_MAX_DEVICES 16

namespace nmrfit {

void count_launches(int n);   // bookkeeping for nmrfit_launch_count()

// Opts `Kernel` into `bytes` of dynamic shared memory on the current device.  The attribute is per device, so it is
// set once per device and kernel (each instantiation of this template keeps its own record).
template <auto Kernel>
cudaError_t opt_in_smem(int bytes) {
    static bool done[NMRFIT_MAX_DEVICES] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (done[dev % NMRFIT_MAX_DEVICES]) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done[dev % NMRFIT_MAX_DEVICES] = true;
    return e;
}

// ---- K1 objective -------------------------------------------------------------
struct ObjArgs {
    const double* spec;     // [B][4][N]: w, u, v, weights
    const double* x;        // [B][S][D] particle positions, D = 4 + 3P
    const double* x_in;     // null, or where the prepare pass READS the positions instead (page-locked host memory mapped
                            // into the device: it copies them to x on the way, each element crossing PCIe once)
    double* partials;       // [B][S][n_tiles][nsum]
    const int* frozen;      // [B] or null: spectra whose swarm has stopped are skipped
    const double* grid_h;   // [B][2] axis spacing h and ulp scale 2^-52*max|w| (uniform-axis kernel only)
    // uniform-axis kernel: per-particle constants written by its prepare pass (see objective_uniform.cu)
    double* prep_coef;      // [B][S][P][8]
    double* prep_part;      // [B][S][68]
    double* prep_far;       // [B][S][n_tiles*nw][sub][kFarPoly = 10]   (tile-major for the streamed kernel)
    double* prep_anchor;    // [B][S][n_tiles*nw][2]
    unsigned* prep_mask;    // [B][S][n_tiles*nw][ceil(P/32)+1]
    int n_tiles, nw;        // point tiles, warps (= regions) per tile (filled by the launcher)
    int N, P, S;
    int kk;                 // 0 real only, 1 reference fit_im (last peak), 2 sum over peaks
    int sp;                 // particles per CTA (filled by the launcher); streamed kernel: particles per pipeline stage
    // streamed uniform-axis kernel (objective_stream.cu): a CTA keeps its point tile and walks `gpc` particle groups
    // through a `stages`-deep pipeline of bulk copies; its prepare pass stores the per-region constants tile-major,
    // [B][n_tiles][S][nw][...], so that one tile's regions of a whole group are one contiguous block
    int tile_major;         // layout of prep_far / prep_anchor / prep_mask (0: [B][S][n_tiles*nw][...])
    int stages, gpc, occ;   // occ: CTAs of 256 threads per SM the streamed kernel is built for (2 or 3)
    int sub;                // far-field cells per region of 32*R points (1, 2 or 4; uniform_eval.cuh); far / mask hold
                            // `sub` entries per region
};

// Calls f(std::integral_constant<int, V>{}) for the V among Vs that equals v, cudaErrorInvalidValue for any other v:
// each launcher lists the values it is built for, and only those are instantiated.
template <int... Vs, typename F>
cudaError_t dispatch(int v, F&& f) {
    cudaError_t e = cudaErrorInvalidValue;
    (void)((v == Vs ? (e = f(std::integral_constant<int, Vs>{}), true) : false) || ...);
    return e;
}
// a plan's threads per CTA (128 | 256) and points per thread (among Rs): f(THREADS, R)
template <int... Rs, typename F>
cudaError_t dispatch_geometry(const ObjTune& t, F&& f) {
    return dispatch<128, 256>(t.threads, [&](auto T) { return dispatch<Rs...>(t.r, [&](auto R) { return f(T, R); }); });
}
// exp table bits of the kernels built for every table
template <typename F>
cudaError_t dispatch_tb(int tb, F&& f) { return dispatch<0, 6, 8, 10>(tb, f); }

struct MoveArgs;
// One objective evaluation as `p` plans it (objective.cu): the stand-alone move of the swarm `mv` or the prepare pass
// (which folds the move in), the evaluation kernel, and the finalize pass when f is set (f == nullptr: the swarm's
// finish kernel sums the tiles itself).  ev0 / evm / ev1 (nullable) are recorded before the first leg, between it and
// the evaluation kernel (at its start on paths without a prepare pass), and after the evaluation kernel.
cudaError_t run_objective_plan(const ObjPlan& p, ObjArgs a, int B, const MoveArgs* mv, double* f, cudaStream_t st,
                               cudaEvent_t ev0, cudaEvent_t evm, cudaEvent_t ev1);

// The evaluation kernel of each file at the plan's geometry (`a` as run_objective_plan fills it)
cudaError_t launch_objective_general(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st);   // objective.cu
cudaError_t launch_objective_uniform(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st);   // objective_uniform.cu
cudaError_t launch_objective_stream(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st);    // objective_stream.cu
cudaError_t launch_objective_f32(const ObjPlan& p, const ObjArgs& a, int B, cudaStream_t st);       // objective_f32.cu
// the prepare pass of the uniform-axis kernels (objective_uniform.cu); mv != nullptr moves the swarm (pso.cu's update)
// in it, one launch fewer per generation
cudaError_t launch_objective_prepare(const ObjPlan& p, const ObjArgs& a, int B, const MoveArgs* mv, cudaStream_t st);

// fixed-order sum over point tiles + sqrt(mean) (shared by the objective kernels)
// `nw` > 1: the partial sums are per REGION, [n_tiles][nw]: the nw regions of a tile are summed first, then the tiles
cudaError_t launch_objective_finalize(const double* partials, int n_tiles, int nsum, int N, int S, int B,
                                      const int* frozen, double* f, cudaStream_t st, int nw = 1);

// ---- K2/K3 swarm --------------------------------------------------------------
struct SwarmState {
    int B, S, D;
    double *x, *v, *p;      // [B][S][D]
    double *fx, *fp;        // [B][S]
    double *g, *fg;         // [B][D], [B]   running global best
    double *best_x, *best_f;// [B][D], [B]   what pso() returns (p_min on an early stop)
    double *lb, *ub;        // [B][D]
    double *rec;            // [B][D+2] local best record: f, global index, position
    int *stop, *it;         // [B] stop reason (0 running), generation counter
    double omega, phip, phig, minstep, minfunc;
    unsigned long long seed;
    long long index0;       // global index of local particle 0 (particle sharding)
    long long spec0;        // global index of local spectrum 0 (spectra sharding)
};

struct MoveArgs {
    SwarmState s;
    const double* rp;       // [B][S][D] host-stream uniforms of this generation, or null for device Philox
    const double* rg;
    int generation;
};
// record exchange over peer memory (pso.cu): device arrays of per-rank window pointers
struct PeerArgs {
    double* const* recs;        // [n_ranks] -> that rank's record window [2][n_ranks][B][D+2]
    long long* const* tokens;   // [n_ranks] -> that rank's token array [n_ranks][B]
    int n_ranks, rank;
    long long token;            // (fit epoch << 32) | generation: monotonic over the life of the windows
    long long max_wait_ns;      // bound of the wait, wall time (%globaltimer)
    int* error;                 // set to 1 when the wait expired
};
// finalize + personal bests + local best record (+ swarm-best commit when `commit`) in one launch:
// partials [B][S][n_tiles][nsum] -> fx, fp, p, rec; `scratch` holds [B][ceil(S/8)][2] doubles, `tickets` [B] zeroed once
cudaError_t launch_swarm_finish(const SwarmState& s, const double* partials, int n_tiles, int nsum, int N, double* rec,
                                double* scratch, unsigned* tickets, int commit, int maxiter, cudaStream_t st, int nw = 1,
                                const PeerArgs* pa = nullptr);   // commit 2 (with pa): exchange over peer memory, then commit
size_t swarm_finish_scratch_doubles(int B, int S);

cudaError_t launch_swarm_exchange_commit(const SwarmState& s, const PeerArgs& pa, int initial, int maxiter,
                                         cudaStream_t st);

cudaError_t launch_swarm_init(const SwarmState& s, const double* r_pos, const double* r_vel, cudaStream_t st);
cudaError_t launch_swarm_init_velocity(const SwarmState& s, const double* r_vel, cudaStream_t st);
cudaError_t launch_swarm_move(const SwarmState& s, const double* rp, const double* rg, int generation, cudaStream_t st);
cudaError_t launch_swarm_commit(const SwarmState& s, const double* recs, int n_ranks, int initial, int maxiter,
                                cudaStream_t st);

// ---- K7 fused swarm generations (swarm_fused.cu) ------------------------------------
struct FusedArgs {
    SwarmState s;
    const double* spec;     // [B][4][N]
    const double* grid_h;   // [B][2]
    const double* rp;       // [n_gen][B][S][D] host-stream uniforms, or null for device Philox
    const double* rg;
    double* rec_f;          // [2][B][S]     published personal-best values, double-buffered by generation parity
    double* rec_x;          // [2][B][S][D]  ... and positions
    unsigned* barrier;      // [B] arrival counters (zeroed by the launcher)
    int N, P;
    int n_vtiles, vw;       // point tiles and warps per tile of the per-step kernels (fixes the summation order)
    int n_gen;              // generations to run in this launch
    int gen0;               // absolute number of the first of them (Philox counter)
    int maxiter;
    int sub;                // far-field cells per region (far_cells_per_region, or the context's override)
    int slots;              // supertiles of (u, v, weights) held in shared memory (filled by the launcher)
    int cluster;            // CTAs (one thread-block cluster) per particle (filled by the launcher)
    int pairs;              // pair-parallel constants pass (needs its scratch in shared memory; filled by the launcher)
    long long* timing;      // optional [8] per-phase cycle counters (null: off)
    int* error;             // raised when the inter-CTA barrier wait expired (a CTA of the spectrum died)
    long long max_wait_ns;  // bound of that wait, wall time
};
struct FusedPlan {
    bool ok, dense, pairs;
    int threads, r, slots, cluster;
    size_t smem;
};
// can B*S CTAs be co-resident for this shape?  plan->ok says so; never launches
// `force`: ignore the size heuristic (NMRFIT_FUSED_REQUIRE)
cudaError_t swarm_fused_plan(const FusedArgs& a, int D, int B, int S, const ObjTune& t, int device, bool force,
                             FusedPlan* plan);
cudaError_t launch_swarm_fused(FusedArgs a, const FusedPlan& plan, int B, int S, cudaStream_t st);

// ---- K8 residual weights of a batch (weights.cu) -----------------------------------
cudaError_t launch_weights(double* spec, double* scratch, const double* bounds_dev, const double* values_dev, int B,
                           int N, int n_windows, int sweeps, double omega, cudaStream_t st);

// ---- K9 phase estimation (phase.cu) --------------------------------------------------
cudaError_t launch_phase_brute(const double* u, const double* v, int B, int N, const double* cands_dev, int K,
                               double* err, int* ok, double* best_p0, double* best_err, cudaStream_t st);
cudaError_t launch_phase_acme(const double* u, const double* v, int B, int N, const double* ph_dev, int K, double* score,
                              cudaStream_t st);

// ---- numpy's legacy MT19937 stream continued on the device (mt19937.cu) --------------------
cudaError_t launch_mt19937(unsigned* key_dev, int* pos_dev, long long n, unsigned* words_dev, double* out_a, double* out_b,
                           long long nsd, cudaStream_t st);

// ---- K10 auto peak selection (peaks.cu) ----------------------------------------------
// front: upsample, smooth, global baseline, maxima (unsorted indices + the upsampled signal there);
// back: per accepted maximum the half-height crossings, local baseline, height, Simpson area
cudaError_t launch_peaks_front(const double* w, const double* u, int B, int N, long long M, const double* sg,
                               double* uu, double* us, double* bmax, int nblk, double* base, int max_it, double tol,
                               long long order, int max_out, long long* maxima, int* n_maxima, double* uu_at_maxima,
                               cudaStream_t st);
cudaError_t launch_peaks_back(const double* w, const double* uu, int B, int N, long long M, const double* base,
                              const long long* pk_i, const double* pk_h, const int* n_pk, int max_peaks, long long* cross,
                              int max_it, double tol, void* out, cudaStream_t st);
cudaError_t launch_peaks_probe(const double* w, int N, long long M, const double* uu, const double* us, int b,
                               const long long* idx, int n, double* out, cudaStream_t st);
size_t peaks_out_bytes();

// ---- K4/K5 curves -------------------------------------------------------------
cudaError_t launch_ps2(const double* u, const double* v, int n, double p0, double p1, int inv, double* re, double* im,
                       cudaStream_t st);
cudaError_t launch_voigt(const double* w, int n, double r, double yoff, double width, double loc, double a, double* out,
                         cudaStream_t st);
cudaError_t launch_kk(const double* w, int n, double r, double width, double loc, double a, double* out,
                      cudaStream_t st);
cudaError_t launch_generate_result(const double* params_host, int P, const double* w, int n, double* real,
                                   double* imag, double* V, double* I, double* u, double* v, cudaStream_t st);

// ---- K12 normal equations of the objective (normal_eq.cu) ---------------------------
// Tiling of the pass: a function of N and P only, so that a spectrum's sums do not depend on the batch.
struct NormalEqPlan {
    int N, P;
    int nb, ep, tri, tasks;     // 4x4 blocks per matrix edge, padded row length, blocks per triangle, both triangles
    int ng, slices, tasks_per_slice, threads;   // point groups per CTA, CTAs per chunk, blocks per CTA, CTA size
    int tp, chunk, n_chunks;    // points per staged tile, points per CTA, chunks per spectrum
    size_t smem;                // dynamic shared memory of the partial kernel, bytes
};
NormalEqPlan normal_eq_plan(int N, int P);
size_t normal_eq_scratch_doubles(const NormalEqPlan& p, int B);
// x [B][D] -> out [B][2*D*D + D + 2] (H, M, g, ssr per spectrum); `part` holds normal_eq_scratch_doubles doubles
cudaError_t launch_normal_eq(const double* spec, const double* x, const NormalEqPlan& p, int B, double* part,
                             double* out, cudaStream_t st);
// K16: the same pass for a robust loss (NMRFIT_LOSS_*; LINEAR is launch_normal_eq), fscale [B] on the device.  Out
// block as launch_normal_eq's with H_rho | M | g_rho | (s_rho, sum w^2 rho' res^2) (normal_eq.cu)
cudaError_t launch_normal_eq_loss(const double* spec, const double* x, int loss, const double* fscale,
                                  const NormalEqPlan& p, int B, double* part, double* out, cudaStream_t st);
// K16 moments of the loss (robust.cu): x [B][D] -> out [B][5]; `part` holds loss_moments_scratch_doubles doubles
size_t loss_moments_scratch_doubles(int B, int N);
cudaError_t launch_loss_moments(const double* spec, const double* x, int loss, const double* fscale, int B, int N,
                                int P, double* part, double* out, cudaStream_t st);
// K17 (scale.cu): x [B][D] -> res [B][N], the residual of K12; res [B][N] -> out [B][2] = (median, MAD), numpy's median
cudaError_t launch_residuals(const double* spec, const double* x, int B, int N, int P, double* res, cudaStream_t st);
cudaError_t launch_median_mad(const double* res, int B, int N, double* out, cudaStream_t st);

// ---- K14 residual autocorrelation and lag-weighted M (lagged.cu) --------------------
// Tiling of both passes: a function of N, P and the largest lag L only.
struct LaggedPlan {
    int N, P, L;
    int nb, ep, tasks;          // 4x4 blocks per edge of M, padded row length, blocks of its upper triangle
    int ng, slices, tasks_per_slice, threads;   // as NormalEqPlan
    int tp, chunk, n_chunks;    // points per tile (staged with L rows of halo on each side), per CTA, chunks
    size_t smem;                // dynamic shared memory of the M partial kernel, bytes
    int max_lag;                // largest L the shared memory holds at this P
    int acf_chunk, acf_n_chunks, acf_threads, acf_segments;   // residual autocorrelation pass: points per CTA,
    size_t acf_smem;                                          // chunks, CTA size, segments of a chunk per lag
};
LaggedPlan lagged_plan(int N, int P, int L);
size_t lagged_m_scratch_doubles(const LaggedPlan& p, int B);
size_t residual_acf_scratch_doubles(const LaggedPlan& p, int B);
// x [B][D] -> r [B][L+1], r_k = sum_{i < N-k} res_i res_{i+k}; `part` holds residual_acf_scratch_doubles doubles
cudaError_t launch_residual_acf(const double* spec, const double* x, const LaggedPlan& p, int B, double* part,
                                double* r, cudaStream_t st);
// x [B][D], rho [B][L+1] -> M [B][D][D] = sum_i sum_{|k| <= L} rho_|k| a_i^T a_{i+k}, a_i = w_i^2 A_i
cudaError_t launch_lagged_m(const double* spec, const double* x, const double* rho, const LaggedPlan& p, int B,
                            double* part, double* M, cudaStream_t st);

// ---- K13 bounded Levenberg-Marquardt refinement on K12 (refine.cu) --------------------
#define NMRFIT_REFINE_RUNNING 0
struct RefineState {
    double lam, f;              // damping of the next trial; sqrt(s/N) at the current point
    int status, passes, accepted, pad;
};
// K15 tie map of a batch (built by nmrfit_ctx_refine_tied): per spectrum the d free parameters theta in index order,
// each with its group G(m) = its master plus its dependents in ascending index.
struct RefineTies {
    const int* ints;        // [B][3D + 2]: d | off [D+1] (G(m) = members off[m] .. off[m+1]) | members [D] | master [D]
    const double* dbls;     // [B][2D]: scale | offset of each member slot (1 | 0 for the master)
};
size_t refine_step_smem(int D);
// trial [B][2*D*D + D + 2] is launch_normal_eq's output at xt; cur [B][D*D + D + 1] holds H | g | s at xc.
// `active` (or null) gains one per spectrum still running after the step.  ties == null: x itself is refined within
// [lb, ub]; else theta within the reduced box [lb, ub] ([B][D], the first d entries of a spectrum's row).
cudaError_t launch_refine_step(const double* trial, double* cur, RefineState* state, double* xc, double* xt,
                               const double* lb, const double* ub, int B, int N, int D, int max_iter, double xtol,
                               int* active, const RefineTies* ties, cudaStream_t st);

// ---- probes -------------------------------------------------------------------
cudaError_t fp64_peak_probe(int iters, int repeats, double* tflops, double* sustained, cudaStream_t st);

}  // namespace nmrfit
