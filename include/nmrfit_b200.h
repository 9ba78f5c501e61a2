/* nmrfit_b200 - C ABI of the B200-native objective-evaluation hot path of pnnl/nmrfit.
 *
 * The reference (pure Python, /root/reference/nmrfit) has no FFI layer of its own;
 * its boundary for this path is the Python call surface
 *     nmrfit.fit(data, lower, upper, ...)                   core.py:64-95
 *     FitUtility.fit / generate_result                      utils.py:164-189, 226-295
 *     pyswarm.pso(objective, lb, ub, args=..., ...)         utils.py:176-182
 *     equations.objective / voigt / kk_relation*            equations.py:152-212, 115-149, 52-112, 242
 *     proc_autophase.ps2                                    proc_autophase.py:9-36
 * Each entry point below names the reference interface it stands in for.  The
 * Python mirror of that surface (the nmrfit_b200 package) binds these symbols with ctypes;
 * INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: pointers and sizes only; no exceptions cross the boundary.
 *   - every function returns NMRFIT_OK (0) or a negative error code; the message
 *     is available from nmrfit_last_error() (thread-local).
 *   - all arrays are float64, C-contiguous.  "dev" = CUDA device memory on the
 *     context's device, "host" = ordinary host memory (pinned or pageable).
 *   - functions taking a `stream` (a cudaStream_t passed as void*, NULL = default
 *     stream) are asynchronous; the caller synchronises.  *_host functions are
 *     synchronous and do their own staging copies.
 *   - the caller owns every buffer it passes; the context owns spectra, swarm
 *     state and scratch.  A context is bound to one device and is not thread-safe.
 *   - D = 4 + 3*n_peaks; a parameter vector is [p0, p1, r, yoff, (width, loc, area) * n_peaks]
 *     (equations.py:177, 188-192).
 */
#ifndef NMRFIT_B200_H
#define NMRFIT_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define NMRFIT_ABI_VERSION 2

#define NMRFIT_OK 0
#define NMRFIT_ERR_ARG (-1)    /* bad argument */
#define NMRFIT_ERR_CUDA (-2)   /* a CUDA call failed */
#define NMRFIT_ERR_STATE (-3)  /* call sequence violated (e.g. spectrum not set) */
#define NMRFIT_ERR_NOMEM (-4)

#define NMRFIT_FP64 0
#define NMRFIT_FP32 1          /* opt-in: FP32 lineshape math, FP64 residual accumulation */

/* objective kernel selection (nmrfit_ctx_set_algorithm) */
#define NMRFIT_ALGO_AUTO 0     /* uniform-axis kernel when every spectrum's w is uniformly spaced, the fit is
                                  real-only and FP64; the general kernel otherwise */
#define NMRFIT_ALGO_GENERAL 1  /* always the general kernel (any w) */
#define NMRFIT_ALGO_UNIFORM 2  /* require the uniform-axis kernel; launches fail with NMRFIT_ERR_STATE if it cannot run */

/* fit_im argument of the objective entry points */
#define NMRFIT_REAL_ONLY 0     /* fit_im is not True: equations.py:202 only */
#define NMRFIT_IM_REFERENCE 1  /* fit_im is True, reference semantics: equations.py:199 overwrites I_fit,
                                  so only the LAST peak's Kramers-Kronig curve enters :206 */
#define NMRFIT_IM_SUM 2        /* imaginary fit accumulated over all peaks (what generate_result does) */

/* stop reasons reported by the swarm (pyswarm's three exits) */
#define NMRFIT_RUNNING 0
#define NMRFIT_STOP_MINFUNC 1
#define NMRFIT_STOP_MINSTEP 2
#define NMRFIT_STOP_MAXITER 3
#define NMRFIT_STOP_PEER_LOST 4   /* particle sharding over peer memory: a peer's record never arrived (error state) */

typedef struct nmrfit_ctx nmrfit_ctx;

int nmrfit_abi_version(void);
const char* nmrfit_last_error(void);
int nmrfit_device_count(int* count);

/* ---- context: one batch of n_spectra spectra of n_points points, n_peaks peaks each ------------- */
int nmrfit_ctx_create(nmrfit_ctx** out, int device, int n_spectra, int n_points, int n_peaks, int precision);
void nmrfit_ctx_destroy(nmrfit_ctx* ctx);

/* Upload spectrum b: the `args=(data.w, data.u, data.v, weights, ...)` tuple of utils.py:176.
 * Host or device pointers (UVA); synchronous. */
int nmrfit_ctx_set_spectrum(nmrfit_ctx* ctx, int b, const double* w, const double* u, const double* v,
                            const double* weights);

/* Bulk form of nmrfit_ctx_set_spectrum: spectra b0 .. b0+count-1 from four [count][n_points] arrays (host or
 * device).  weights may be NULL when nmrfit_ctx_compute_weights follows. */
int nmrfit_ctx_set_spectra(nmrfit_ctx* ctx, int b0, int count, const double* w, const double* u, const double* v,
                           const double* weights);

/* FitUtility._compute_weights (utils.py:191-224) + equations.laplace1d (equations.py:215-238) for every spectrum of
 * the context at once, written into the context's weights plane: windows [argmin|w-b0|, argmin|w-b1|] per peak,
 * later peaks overwriting earlier ones, then `sweeps` Jacobi sweeps with pinned ends (reference: 10, omega
 * 0.33333333).  peak_bounds [n_spectra][n_windows][2] = Peak.bounds; peak_values [n_spectra][n_windows] =
 * (max|height| / |height_k|)**expon, computed by the caller.  weights_out: optional [n_spectra][n_points] copy
 * (host or device).  Bit-identical to the reference's numpy result. */
int nmrfit_ctx_compute_weights(nmrfit_ctx* ctx, const double* peak_bounds, const double* peak_values, int n_windows,
                               int sweeps, double omega, double* weights_out, void* stream);

/* Normal equations of the objective at one parameter vector per spectrum, from the spectra and weights the context
 * holds (any axis; FP64 on FP32 contexts too).  With D = 4 + 3P, x = [p0, p1, r, yoff, (width, loc, area) x P],
 *   res_i = Vdata_i(p0, p1) - Vfit_i(x),   Vdata = Re ps2(u, v, p0, p1),   Vfit = sum_k [yoff + a_k (r L_k + (1-r) G_k)]
 * and A_i = d res_i / dx (d/dp0 = -Idata_i, d/dp1 = -Idata_i * i/N, d/dyoff = -P, d/dr = -sum_k a_k (L_k - G_k),
 * d/da_k = -(r L_k + (1-r) G_k), and the closed-form width and location derivatives), over all n_points:
 *   H = sum w_i^2 A_i^T A_i,  M = sum w_i^4 A_i^T A_i,  g = sum w_i^2 res_i A_i,  ssr = (sum w_i^2 res_i^2, sum res_i^2)
 * where w_i are the weights.  x [n_spectra][D]; H, M [n_spectra][D][D] (both triangles), g [n_spectra][D],
 * ssr [n_spectra][2].  Host or device pointers (UVA); any output may be NULL; returns when the outputs are written.
 * Sums are in a fixed order that depends on n_points and n_peaks only: bit-reproducible, and a spectrum's result
 * is the same alone or in a batch.  n_peaks <= 64; NMRFIT_ERR_ARG above. */
int nmrfit_ctx_normal_equations(nmrfit_ctx* ctx, const double* x, double* H, double* M, double* g, double* ssr,
                                void* stream);
/* The launch plan nmrfit_ctx_normal_equations uses for n_points points and n_peaks peaks (host only, no CUDA call).
 * out[10] = point groups per CTA, task slices per chunk, 4x4 blocks of both triangles (tasks), tasks per slice, threads
 * per CTA, points per staged tile, points per chunk, chunks, dynamic shared memory (bytes), scratch doubles per spectrum.
 * NMRFIT_ERR_ARG unless 1 <= n_peaks <= 64 and n_points >= 1. */
int nmrfit_normal_eq_plan(int n_points, int n_peaks, int* out);

/* Correlated noise (DESIGN K14), from the spectra and weights the context holds, at one x [n_spectra][D] per spectrum,
 * with res_i and A_i as in nmrfit_ctx_normal_equations and L = max_lag:
 *   nmrfit_ctx_residual_acf:    r_out [n_spectra][L+1],  r_k = sum_{i=0}^{N-1-k} res_i res_{i+k}  (r_0 = ssr[1]);
 *   nmrfit_ctx_normal_m_lagged: M_out [n_spectra][D][D] = sum_i sum_{|k| <= L, 0 <= i+k < N} rho_|k| a_i^T a_{i+k},
 *                               a_i = w_i^2 A_i, from rho [n_spectra][L+1]  (L = 0, rho = 1: the M of K12).
 * Host or device pointers; they return when the outputs are written.  Sums are in a fixed order that depends on
 * n_points, n_peaks and L only: bit-reproducible, the same alone or in a batch; M_out is exactly symmetric.
 * NMRFIT_ERR_ARG for NULL pointers, more than 64 peaks, max_lag < 0, max_lag >= n_points, max_lag above the cap of
 * nmrfit_lagged_plan, or a non-finite rho. */
int nmrfit_ctx_residual_acf(nmrfit_ctx* ctx, const double* x, int max_lag, double* r_out, void* stream);
int nmrfit_ctx_normal_m_lagged(nmrfit_ctx* ctx, const double* x, const double* rho, int max_lag, double* M_out,
                               void* stream);
/* The launch plan of both lagged passes (host only, no CUDA call).  out[14] = point groups per CTA, task slices per
 * chunk, 4x4 blocks of the upper triangle (tasks), tasks per slice, threads per CTA, points per staged tile, points per
 * chunk, chunks, dynamic shared memory (bytes), scratch doubles per spectrum (M pass); the largest max_lag at n_peaks;
 * points per chunk, chunks and scratch doubles per spectrum of the residual pass.  NMRFIT_ERR_ARG unless
 * 1 <= n_peaks <= 64, n_points >= 1 and 0 <= max_lag <= the cap (query max_lag = 0 to learn the cap). */
int nmrfit_lagged_plan(int n_points, int n_peaks, int max_lag, int* out);

/* How nmrfit_ctx_refine left a spectrum. */
#define NMRFIT_REFINE_CONVERGED 1   /* an accepted step was at most xtol of every parameter's diagonal noise scale */
#define NMRFIT_REFINE_STALLED 2     /* the damping passed 1e16 without a descent step: a numerical minimum */
#define NMRFIT_REFINE_MAX_ITER 3    /* max_iter passes of the normal equations */
#define NMRFIT_REFINE_NONFINITE 4   /* H, g or s is not finite at the start; x is left as it was */

/* Bounded Levenberg-Marquardt refinement of one parameter vector per spectrum to the least-squares optimum of the
 * weighted residual (DESIGN K13), from the spectra and weights the context holds, looping on the device.  Each pass
 * forms the normal equations at a trial point (as nmrfit_ctx_normal_equations does); one CTA per spectrum accepts the
 * trial if its s = sum w^2 res^2 is finite and strictly below the current one, updates the damping lam (1e-3 at the
 * start; /10 down to 1e-12 on acceptance, *10 on rejection), and solves (S H S + lam I) y = -S g, S = diag(H_jj^-1/2),
 * over the parameters not frozen (H_jj = 0, or at a bound with the gradient pointing out), for the next trial
 * clip(x + S y, lb, ub).  A spectrum stops CONVERGED when an accepted step has max_j |dx_j| sqrt(H_jj (N-D)/s) <= xtol
 * (H and s of the point the step was built from), or STALLED, MAX_ITER (max_iter passes, counting the one at the start)
 * or NONFINITE.  x_inout [n_spectra][D]: the start in, the refined point out (bit for bit the start if no step was
 * accepted); lb, ub [n_spectra][D]; f_out = sqrt(s/N) at the returned point, passes_out, accepted_out, status_out
 * [n_spectra] (any of the four may be NULL).  Host or device pointers; returns when the outputs are written.  The
 * result of a spectrum is bit-reproducible and the same alone or in a batch, on FP32 contexts too.  NMRFIT_ERR_ARG for
 * more than 64 peaks, n_points <= D, lb_j >= ub_j, a start outside its box, max_iter < 1 or xtol <= 0. */
int nmrfit_ctx_refine(nmrfit_ctx* ctx, double* x_inout, const double* lb, const double* ub, int max_iter, double xtol,
                      double* f_out, int* passes_out, int* accepted_out, int* status_out, void* stream);

/* nmrfit_ctx_refine with fixed and linked parameters (DESIGN K15).  tie_master, tie_scale, tie_offset [n_spectra][D]
 * give each parameter j of a spectrum one of three roles:
 *   free    tie_master[j] = j;
 *   fixed   tie_master[j] = -1: x_j = tie_offset[j];
 *   linked  tie_master[j] = k != j, k free: x_j = tie_scale[j] * x_k + tie_offset[j] (no chains).
 * Scale and offset are read for linked parameters (scale finite and non-zero, offset finite) and the offset for fixed
 * ones (finite); the box of a fixed parameter is not read.  The d free parameters theta, in index order, are refined
 * as nmrfit_ctx_refine refines x, within the reduced box: the master's own box intersected with each dependent's box
 * mapped through its tie, [(lb_j - c_j)/a_j, (ub_j - c_j)/a_j] (swapped for a_j < 0).  H and g of theta are
 * H_theta[m][n] = sum_{j in G(m)} sum_{k in G(n)} a_j a_k H_jk and g_theta[m] = sum_{j in G(m)} a_j g_j, G(m) the master
 * (a = 1) and its dependents in ascending index, summed in that order without FMA (the identity map gives H and g
 * exactly); the convergence test uses H_theta and N - d.  A trial is expanded as x_j = a_j * theta_m + c_j rounded
 * twice, so numpy's `a * t + c` gives the same bits; dependents are not clipped to their own box and leave it at a
 * reduced bound only by that rounding.  The start: free entries of x_inout are clipped into the reduced box (NaN to
 * its lower end), the others are recomputed by the expansion; no start is refused.  Outputs as nmrfit_ctx_refine, x
 * expanded.  Spectra of one batch may carry different maps.  NMRFIT_ERR_ARG, with the spectrum and parameter named, for
 * a master out of [-1, D), a chain (a master that is itself linked), a fixed master, a zero or non-finite scale, a
 * non-finite offset, an empty or single-point reduced box, n_points <= d, and for what nmrfit_ctx_refine refuses
 * besides the box and the start. */
int nmrfit_ctx_refine_tied(nmrfit_ctx* ctx, double* x_inout, const double* lb, const double* ub, const int* tie_master,
                           const double* tie_scale, const double* tie_offset, int max_iter, double xtol, double* f_out,
                           int* passes_out, int* accepted_out, int* status_out, void* stream);

/* Robust losses of the refinement (DESIGN K16), in scipy.optimize.least_squares' convention: with the unweighted
 * residual res_i, the scale c = f_scale > 0 of its spectrum (units of the data u) and z_i = (res_i / c)^2,
 *   LINEAR  rho(z) = z                       (least squares: the paths above, bit for bit)
 *   HUBER   rho(z) = z for z <= 1, else 2 sqrt(z) - 1
 *   SOFT_L1 rho(z) = 2 (sqrt(1 + z) - 1)
 *   CAUCHY  rho(z) = ln(1 + z)
 * The loss is per call; the scale is per spectrum, since the spectra of one batch have different noise levels. */
#define NMRFIT_LOSS_LINEAR 0
#define NMRFIT_LOSS_HUBER 1
#define NMRFIT_LOSS_SOFT_L1 2
#define NMRFIT_LOSS_CAUCHY 3

/* Robust normal equations at one x [n_spectra][D] per spectrum, with res_i, A_i and w_i as in
 * nmrfit_ctx_normal_equations and rho' = d rho / dz > 0:
 *   H [n_spectra][D][D] = sum w_i^2 rho'(z_i) A_i^T A_i   (the Gauss-Newton matrix of iteratively reweighted LS)
 *   g [n_spectra][D]    = sum w_i^2 rho'(z_i) res_i A_i   (the gradient of cost / 2)
 *   cost [n_spectra]    = sum w_i^2 c^2 rho(z_i)
 * One pass of K12's launch plan, each point's row of H_ext scaled by sqrt(rho'); any output may be NULL.  With
 * NMRFIT_LOSS_LINEAR the outputs are nmrfit_ctx_normal_equations' H, g and ssr[0] bit for bit and f_scale is not read.
 * Host or device pointers; returns when the outputs are written; fixed summation order (as K12).  NMRFIT_ERR_ARG for a
 * NULL x, an unknown loss, more than 64 peaks, and for a non-linear loss a NULL f_scale or one that is not finite and
 * > 0 (the message names the spectrum). */
int nmrfit_ctx_normal_equations_loss(nmrfit_ctx* ctx, const double* x, int loss, const double* f_scale, double* H,
                                     double* g, double* cost, void* stream);
/* The moments of the loss at one x [n_spectra][D] per spectrum, out [n_spectra][5] =
 *   (cost = sum w_i^2 c^2 rho(z_i),  sum w_i^2 res_i^2,  sum psi_i^2,  sum psi'_i,  sum psi'_i^2)
 * with psi_i = rho'(z_i) res_i and psi'_i = rho'(z_i) + 2 z_i rho''(z_i) (unweighted: they give the M-estimator's scale
 * factor of the sandwich covariance, DESIGN K16).  For LINEAR psi = res, psi' = 1 and f_scale is not read.  Chunk
 * partials added in a fixed order: bit-reproducible, the same alone or in a batch.  Refusals as
 * nmrfit_ctx_normal_equations_loss, and a NULL out. */
int nmrfit_ctx_loss_moments(nmrfit_ctx* ctx, const double* x, int loss, const double* f_scale, double* out,
                            void* stream);
/* nmrfit_ctx_refine (tie arrays NULL) or nmrfit_ctx_refine_tied (all three given) on the robust cost: every pass is
 * nmrfit_ctx_normal_equations_loss at the trial, and the step kernel runs its rules unchanged on (H, g, cost) of the
 * loss: acceptance on the cost, damping, frozen set, statuses, and convergence max |dx_j| sqrt(H_jj (N - d)/cost) <= xtol.
 * f_out = sqrt(cost / N) at the returned point.  With NMRFIT_LOSS_LINEAR the outputs are those of nmrfit_ctx_refine /
 * nmrfit_ctx_refine_tied bit for bit and f_scale is not read.  NMRFIT_ERR_ARG for what those refuse, an unknown loss,
 * tie arrays given only in part, and for a non-linear loss a NULL f_scale or one not finite and > 0 (naming the
 * spectrum). */
int nmrfit_ctx_refine_loss(nmrfit_ctx* ctx, double* x_inout, const double* lb, const double* ub, const int* tie_master,
                           const double* tie_scale, const double* tie_offset, int loss, const double* f_scale,
                           int max_iter, double xtol, double* f_out, int* passes_out, int* accepted_out,
                           int* status_out, void* stream);

/* The residual scale (DESIGN K17), from the spectra the context holds, at one x [n_spectra][D] per spectrum, with
 * res_i the unweighted residual of nmrfit_ctx_normal_equations over all n_points points:
 *   nmrfit_ctx_residuals:      res_out [n_spectra][n_points] = res;
 *   nmrfit_ctx_residual_scale: out [n_spectra][2] = (med, MAD), med = median(res) and MAD = median(|res - med|), each
 *                              the value numpy's median gives (the middle order statistic, or (a + b) / 2 of the two
 *                              middle ones for an even count; NaN for a row holding a NaN; -0 and +0 compare equal).
 * The normal-consistent noise level is sigma = MAD / 0.6744897501960817 (the standard normal quantile at 3/4), as
 * scipy.stats.median_abs_deviation(res, scale='normal').  Both run in FP64 on FP32 contexts too, and the selection is
 * exact: the result is the same alone or in a batch and from call to call.  Host or device pointers; they return
 * when the outputs are written.  NMRFIT_ERR_ARG for NULL pointers and more than 64 peaks. */
int nmrfit_ctx_residuals(nmrfit_ctx* ctx, const double* x, double* res_out, void* stream);
int nmrfit_ctx_residual_scale(nmrfit_ctx* ctx, const double* x, double* out, void* stream);

/* Which objective kernel runs (default NMRFIT_ALGO_AUTO), and which one a launch with this fit_im would use.
 * Both kernels evaluate equations.objective (equations.py:152-212); the uniform-axis one exploits
 * w_i = w_0 + i*h (what core.load builds, core.py:58-60) to replace most exponentials by a recurrence. */
int nmrfit_ctx_set_algorithm(nmrfit_ctx* ctx, int algorithm);
int nmrfit_ctx_get_algorithm(nmrfit_ctx* ctx, int fit_im, int* algorithm);

/* Launch geometry of the objective kernel; 0 keeps the automatic choice for that field.
 * threads in {128, 256}; points_per_thread in {2, 4, 8} (general kernel) or {4, 8, 16} (uniform-axis
 * kernel); exp_table_bits in {-1 (no table), 6, 8, 10}.  nmrfit_ctx_get_tuning reports the geometry that runs for a
 * real-only call of n_particles: FP32 contexts run 4 or 8 points per thread on a uniform axis (16 runs as 8) and
 * 256 threads x 4 points on any other axis. */
int nmrfit_ctx_set_tuning(nmrfit_ctx* ctx, int threads, int points_per_thread, int exp_table_bits,
                          int particles_per_cta);
int nmrfit_ctx_get_tuning(nmrfit_ctx* ctx, int n_particles, int* threads, int* points_per_thread, int* exp_table_bits,
                          int* particles_per_cta, int* n_point_tiles);
/* Which FP64 uniform-axis evaluation kernel runs (development / A-B measurement knob; results are bit-identical):
 * variant -1 the library's choice (the streamed kernel), 0 one particle group per CTA (objective_uniform_kernel),
 * 1 streamed (objective_stream_kernel: a CTA keeps its point tile and walks many particle groups through a
 * `stages`-deep ring of TMA-filled shared-memory slots; stages 0 = auto, else 2..4; occupancy 0 = auto, else 2 or 3
 * CTAs of 256 threads per SM - 2 trades resident warps for shared memory and registers). */
int nmrfit_ctx_set_variant(nmrfit_ctx* ctx, int variant, int stages, int occupancy);
int nmrfit_ctx_get_variant(nmrfit_ctx* ctx, int n_particles, int* variant, int* stages);
/* Far-field cells per region of 32 * points_per_thread points (csrc/uniform_eval.cuh): 0 = the library's rule (a
 * function of the axis length only: 64-point cells below 8,192 points, 128-point cells below 32,768, else the whole
 * region), or 1, 2, 4.  Every FP64 uniform-axis kernel of the context follows it; results agree to rounding. */
int nmrfit_ctx_set_far_cells(nmrfit_ctx* ctx, int cells);

/* Small swarms: nmrfit_pso_run executes its generations in ONE cooperative launch (one CTA - on longer axes one
 * thread-block cluster of up to 8 CTAs exchanging through distributed shared memory - per particle, one barrier per
 * generation) instead of three launches per generation - the loop pyswarm.pso runs on the host
 * (call site utils.py:176-182).  Bit-identical to the per-step kernels.  AUTO uses it whenever it can run
 * (FP64, uniform axis, real-only fit, n_spectra * swarmsize CTAs co-resident); REQUIRE makes nmrfit_pso_run
 * fail with NMRFIT_ERR_STATE otherwise. */
#define NMRFIT_FUSED_AUTO 0
#define NMRFIT_FUSED_OFF 1
#define NMRFIT_FUSED_REQUIRE 2
int nmrfit_ctx_set_fused(nmrfit_ctx* ctx, int mode);
int nmrfit_ctx_fused_launches(nmrfit_ctx* ctx, long long* launches);
/* Measurement hook: when enabled, CTA 0 of the fused kernel adds up the SM clock cycles of each phase of a generation
 * (move, constants, objective, tile sums, publish, barrier, argmin, commit).  cycles (nullable): read the 8 counters
 * accumulated so far before they are reset. */
int nmrfit_ctx_fused_timing(nmrfit_ctx* ctx, int enable, long long* cycles);

/* Per-launch timing of the objective kernel with CUDA events on the launching stream (for bench.py's
 * roofline: enable, run, then read the summed duration and the launch count; read resets). */
int nmrfit_ctx_profile(nmrfit_ctx* ctx, int enable);
int nmrfit_ctx_profile_read(nmrfit_ctx* ctx, double* total_ms, long long* launches);
/* The same, split at the event recorded between the two passes of the uniform-axis path: per-particle constants
 * (prepare kernel, with the swarm's move when it is folded in) and the evaluation kernel proper - the roofline's
 * dominant kernel.  Paths without a prepare pass report 0 for it. */
int nmrfit_ctx_profile_read_split(nmrfit_ctx* ctx, double* prepare_ms, double* evaluate_ms, long long* launches);

/* ---- objective: equations.objective (equations.py:152-212) for a whole swarm generation -------
 * x [n_spectra][n_particles][D] -> f [n_spectra][n_particles].  One call replaces the
 * n_particles Python callbacks pyswarm makes per generation (utils.py:176-182). */
int nmrfit_objective_batch(nmrfit_ctx* ctx, const double* x_dev, int n_particles, int fit_im, double* f_dev,
                           void* stream);
int nmrfit_objective_batch_host(nmrfit_ctx* ctx, const double* x_host, int n_particles, int fit_im, double* f_host);
/* equations.objective(x, w, u, v, weights) as the reference calls it - the spectrum comes along with every call - for a
 * context of ONE spectrum: set_spectrum + objective_batch_host in one.  An unchanged spectrum is not sent again; with
 * page-locked positions the kernels are launched before the arrays are compared with the context's host copy (the
 * comparison overlaps the evaluation; a spectrum that did change is uploaded and the evaluation repeated). */
int nmrfit_objective_spectrum_host(nmrfit_ctx* ctx, const double* w, const double* u, const double* v,
                                   const double* weights, const double* x_host, int n_particles, int fit_im,
                                   double* f_host);

/* ---- swarm: pyswarm.pso as called at utils.py:176-182, state resident on the device -----------
 * Generation g (g = 0 is the initial swarm) is   begin|advance -> [exchange records] -> commit.
 * With one rank the exchange is skipped (commit with recs_dev = NULL). */
typedef struct nmrfit_pso_opts {
    int swarmsize;               /* particles held by THIS context (local shard) */
    int maxiter;
    double omega, phip, phig;    /* utils.py:179-181 defaults -0.2134, -0.3344, 2.3259 */
    double minstep, minfunc;     /* pyswarm defaults 1e-8, never overridden by the reference */
    int fit_im;                  /* NMRFIT_REAL_ONLY | NMRFIT_IM_REFERENCE | NMRFIT_IM_SUM */
    int bounds_per_spectrum;     /* 0: lb/ub are [D] shared by all spectra; 1: [n_spectra][D] */
    unsigned long long seed;     /* device Philox stream, used wherever a random array is NULL */
    long long particle_offset;   /* global index of local particle 0 (particle sharding; else 0) */
    long long spectrum_offset;   /* global index of local spectrum 0 (spectra sharding; else 0): with both offsets the
                                    device random stream does not depend on how the work is split over ranks */
} nmrfit_pso_opts;

/* Initial swarm: x = lb + r_pos*(ub-lb), v = vlow + r_vel*(vhigh-vlow), evaluate, personal bests,
 * local best record.  lb/ub: host.  r_pos/r_vel: [n_spectra][swarmsize][D] uniforms in [0,1), host or
 * device, or NULL for device Philox. */
int nmrfit_pso_begin(nmrfit_ctx* ctx, const double* lb, const double* ub, const nmrfit_pso_opts* opts,
                     const double* r_pos, const double* r_vel, void* stream);
/* One generation: velocity/position update with rp, rg (host, device, or NULL = Philox), clamp to the
 * box, evaluate, personal bests, local best record. */
int nmrfit_pso_advance(nmrfit_ctx* ctx, const double* rp, const double* rg, void* stream);
/* One whole generation of a swarm held by ONE context (no rank exchange): advance + commit, asynchronous on `stream` -
 * what nmrfit_pso_run does per generation, without its final synchronisation.  Three launches. */
int nmrfit_pso_step(nmrfit_ctx* ctx, const double* rp, const double* rg, void* stream);
/* ---- numpy's legacy random stream, continued on the device (csrc/mt19937.cu) -----------------------------------
 * pyswarm draws from numpy's global MT19937 (rand(S, D) twice, then uniform(size=(S, D)) twice per generation; call site
 * utils.py:176-182).  Instead of drawing those arrays on the host and copying them, hand over the generator's state
 * (np.random.get_state(): key [624], pos): the device produces the next n_arrays arrays of `elements_per_array`
 * doubles exactly as RandomState.random_sample does, de-interleaved into two device buffers owned by the context
 * (arrays 0, 2, 4, ... -> *a_dev, arrays 1, 3, 5, ... -> *b_dev: positions / velocities, or rp / rg per generation),
 * and returns the advanced state (np.random.set_state) - bit-identical numbers, the stream left where pyswarm would
 * have left it.  The pointers are valid until the next call and may be passed to nmrfit_pso_begin / nmrfit_pso_run. */
int nmrfit_ctx_mt19937_shape(nmrfit_ctx* ctx, long long elements_per_array);
int nmrfit_ctx_mt19937(nmrfit_ctx* ctx, unsigned* key, int* pos, long long n_arrays, double** a_dev, double** b_dev,
                       void* stream);
/* The same in two halves on a stream of the context's own: `begin` queues the generation (state: key [624], pos) and
 * returns at once; `end` waits for it and returns the advanced state (key_out / pos_out nullable: a draw that turns out
 * not to be needed is simply dropped).  Meanwhile the caller runs the swarm on the arrays of the previous begin - the
 * sequential recurrence hides behind the fit's kernels.  Two sets of arrays are used in turn: the pointers of one begin
 * stay valid until the begin after the next. */
int nmrfit_ctx_mt19937_begin(nmrfit_ctx* ctx, const unsigned* key, int pos, long long n_arrays, double** a_dev,
                             double** b_dev);
int nmrfit_ctx_mt19937_end(nmrfit_ctx* ctx, unsigned* key_out, int* pos_out);

/* ---- particle sharding without a collective call: the record exchange over peer memory (NVLink stores) -----------
 * Each rank's context owns a window of records and generation tokens; every rank maps every window (CUDA IPC between
 * processes, plain pointers between contexts of one process).  nmrfit_pso_commit_peers replaces "all-gather the records,
 * nmrfit_pso_commit": one kernel stores this rank's record into every peer's window, publishes the generation token,
 * waits (bounded in wall time) for all ranks' tokens and commits.  nmrfit_pso_step_peers is a whole sharded generation
 * with that exchange folded into the finish kernel's last CTA: the same THREE launches as an unsharded generation and no
 * NCCL call; nmrfit_pso_run_peers runs a chunk of generations in one call (no per-generation host round trip) and
 * synchronises.  Same results as the all-gather path, bit for bit.  On a timeout (nmrfit_pso_peer_timeout, default 20 s)
 * the rank raises its error flag and marks the spectrum stopped with NMRFIT_STOP_PEER_LOST; the other ranks then time
 * out one generation later.  The caller makes the failure collective (swarm.pso_sharded all-reduces the flag).
 *   export: allocate the window for n_ranks; ipc_handle_out (64 bytes, nullable) for other processes, base_out
 *           (nullable) for other contexts of this process.
 *   open:   ipc_handles [n_ranks][64] and/or local_bases [n_ranks] (entry `rank` is ignored).
 *   error:  1 when a wait expired (a peer never arrived); the swarm state is then undefined. */
int nmrfit_pso_peer_export(nmrfit_ctx* ctx, int n_ranks, int rank, void* ipc_handle_out, void** base_out);
int nmrfit_pso_peer_open(nmrfit_ctx* ctx, const void* ipc_handles, void* const* local_bases);
int nmrfit_pso_commit_peers(nmrfit_ctx* ctx, void* stream);
int nmrfit_pso_step_peers(nmrfit_ctx* ctx, const double* rp, const double* rg, void* stream);
int nmrfit_pso_run_peers(nmrfit_ctx* ctx, int n_generations, const double* rp_all, const double* rg_all, int* n_running,
                         int* timed_out, void* stream);
int nmrfit_pso_peer_timeout(nmrfit_ctx* ctx, double milliseconds);
int nmrfit_pso_peer_error(nmrfit_ctx* ctx, int* timed_out);
/* The same exchange for a C consumer WITHOUT a collective library: n contexts of ONE process, one per GPU (or several
 * on one GPU), form a communicator.  This is the library-level counterpart of the reference's `processes=N`
 * (utils.py:182: pyswarm farms the objective calls of a generation out to a multiprocessing pool) - here the
 * particles of the swarm are split over the contexts instead.
 *   init_all: allocates every context's window, enables peer access between their devices and maps every window into
 *             every context (rank = position in ctxs).  Call before nmrfit_pso_begin; each context then begins its own
 *             shard (nmrfit_pso_opts.particle_offset = first global particle index of the shard).
 *   commit:   the initial swarm-best selection over all shards (after every context's nmrfit_pso_begin).
 *   run:      n_generations sharded generations on every context (three launches per context and generation, queued
 *             rank by rank so that no rank's host call waits for another), then one synchronisation.  rp_all / rg_all:
 *             per-context host or device arrays [n_generations][particles of the shard][D], or NULL for the device
 *             random stream.  n_running: spectra not yet stopped; timed_out: 1 if a rank was lost. */
int nmrfit_comm_init_all(nmrfit_ctx* const* ctxs, int n);
int nmrfit_comm_commit(nmrfit_ctx* const* ctxs, int n);
int nmrfit_comm_run(nmrfit_ctx* const* ctxs, int n, int n_generations, const double* const* rp_all,
                    const double* const* rg_all, int* n_running, int* timed_out);
/* Device pointer and length (doubles) of the local best record, [n_spectra][D+2] = (f, global index, x[D]). */
int nmrfit_pso_record(nmrfit_ctx* ctx, double** rec_dev, int* n_doubles);
/* Swarm-best update and the minfunc/minstep/maxiter tests.  recs_dev = [n_ranks][n_spectra][D+2]
 * gathered records (rank order), or NULL to commit this context's own record (n_ranks ignored). */
int nmrfit_pso_commit(nmrfit_ctx* ctx, const double* recs_dev, int n_ranks, void* stream);
/* Run up to n_generations generations on one rank (advance+commit each).  rp_all/rg_all:
 * [n_generations][n_spectra][swarmsize][D] host or device arrays, or NULL for Philox.  Synchronises and
 * returns in *n_running how many spectra have not stopped. */
int nmrfit_pso_run(nmrfit_ctx* ctx, int n_generations, const double* rp_all, const double* rg_all, int* n_running,
                   void* stream);
/* Result (synchronises): x_best [n_spectra][D], f_best [n_spectra], generations done, stop reason.
 * On a minfunc/minstep stop this is (p_min, fp[i_min]) exactly as pyswarm returns it. Any pointer may be NULL. */
int nmrfit_pso_get_best(nmrfit_ctx* ctx, double* x_best, double* f_best, int* generations, int* stop_reason);
/* Copy swarm arrays to the host for inspection; any pointer may be NULL. x,v,p: [n_spectra][swarmsize][D]; fx,fp: [..][swarmsize] */
int nmrfit_pso_get_state(nmrfit_ctx* ctx, double* x, double* v, double* p, double* fx, double* fp);

/* ---- curves ----------------------------------------------------------------------------------- */
/* proc_autophase.ps2 (proc_autophase.py:9-36) */
int nmrfit_ps2(const double* u_dev, const double* v_dev, int n, double p0, double p1, int inv, double* re_dev,
               double* im_dev, void* stream);
int nmrfit_ps2_host(int device, const double* u, const double* v, int n, double p0, double p1, int inv, double* re,
                    double* im);
/* equations.voigt (equations.py:115-149) */
int nmrfit_voigt(const double* w_dev, int n, double r, double yoff, double width, double loc, double a,
                 double* out_dev, void* stream);
int nmrfit_voigt_host(int device, const double* w, int n, double r, double yoff, double width, double loc, double a,
                      double* out);
/* equations.kk_relation_vectorized / kk_relation_parallel (equations.py:52-112, 242), closed form */
int nmrfit_kk(const double* w_dev, int n, double r, double yoff, double width, double loc, double a, double* out_dev,
              void* stream);
int nmrfit_kk_host(int device, const double* w, int n, double r, double yoff, double width, double loc, double a,
                   double* out);
/* FitUtility.generate_result (utils.py:243-295) on the grid w[n]: real/imag [n_peaks][n], V/I/u/v [n].
 * params: host, D doubles. */
int nmrfit_generate_result(const double* params, int n_peaks, const double* w_dev, int n, double* real_dev,
                           double* imag_dev, double* V_dev, double* I_dev, double* u_dev, double* v_dev,
                           void* stream);
int nmrfit_generate_result_host(int device, const double* params, int n_peaks, const double* w, int n, double* real,
                                double* imag, double* V, double* I, double* u, double* v);

/* ---- measurement ------------------------------------------------------------------------------ */
/* ---- phase estimation before the fit: Data.shift_phase(method='brute' | 'auto') (containers.py:51-78) for a batch
 * of spectra.  The handle keeps device copies of u, v ([n_spectra][n_points], host or device source). */
typedef struct nmrfit_phase nmrfit_phase;
int nmrfit_phase_create(nmrfit_phase** out, int device, int n_spectra, int n_points, const double* u, const double* v);
void nmrfit_phase_destroy(nmrfit_phase* h);
/* Data._brute_phase (containers.py:98-110): p0_candidates [K] = np.arange(-pi, pi, step); best_p0 [n_spectra] (0 when
 * no candidate points upwards, as in the reference); optional best_err [n_spectra], err [n_spectra][K], ok
 * [n_spectra][K].  All host pointers. */
int nmrfit_phase_brute(nmrfit_phase* h, const double* p0_candidates, int K, double* best_p0, double* best_err,
                       double* err, int* ok);
/* _ps_acme_score (proc_autophase.py:142-187) for K candidates ph [K][2] = (p0, p1) in RADIANS (the reference's ps()
 * converts its degree arguments first, proc_autophase.py:60-62) -> score [n_spectra][K].  Host pointers. */
int nmrfit_phase_acme(nmrfit_phase* h, const double* ph, int K, double* score);

/* ---- automatic peak selection for a batch of spectra (csrc/peaks.cu) ------------------------------------------
 * Replaces utils.AutoPeakSelector (utils.py:670-783; reached through Data.select_peaks('auto'), containers.py:159-161):
 * linear upsampling onto np.linspace(w.min(), w.max(), upsample * n_points) (utils.py:711-714), Savitzky-Golay(11, 4)
 * smoothing (:716), peakutils.baseline(., 0) (:718), scipy.signal.argrelmax with a window of `window` axis units (:728-733)
 * and, per maximum, half-height crossings, +-2-width bounds, local baseline, height and Simpson area (:747-770).
 *   maxima:  w, u [n_spectra][n_points] (host or device), w ASCENDING (interp1d sorts its input; the caller mirrors that).
 *            sg_coeffs (nullable): 11 smoothing coefficients + the two [5][11] edge maps (tools/gen_sg.py).
 *            Out: n_maxima [n_spectra]; maxima [n_spectra][max_peaks] upsampled indices in NO particular order; the
 *            upsampled signal there; the global baseline [n_spectra].  NMRFIT_ERR_STATE if a spectrum has more.
 *   measure: the caller sorts the maxima, forms height = uu - baseline, applies the threshold (utils.py:735-738) and hands
 *            the survivors back: n_peaks [n_spectra], peak_i / peak_height [n_spectra][max_peaks].  Out, same shape:
 *            ok (1 kept, 0 dropped by x_left < x_right at utils.py:755, -1 no crossing found: the reference raises),
 *            loc, width, bounds [..][2], local_baseline, height, area, idx_range [..][2] (first / last sample in bounds).
 *   probe:   upsampled axis, signal and smoothed signal of spectrum b at n indices (for tests). */
typedef struct nmrfit_peaks nmrfit_peaks;
int nmrfit_peaks_create(nmrfit_peaks** out, int device, int n_spectra, int n_points, int upsample, int max_peaks);
void nmrfit_peaks_destroy(nmrfit_peaks* h);
int nmrfit_peaks_maxima(nmrfit_peaks* h, const double* w, const double* u, double window, const double* sg_coeffs,
                        int baseline_max_it, double baseline_tol, int* n_maxima, long long* maxima, double* uu_at_maxima,
                        double* baseline);
int nmrfit_peaks_measure(nmrfit_peaks* h, const int* n_peaks, const long long* peak_i, const double* peak_height,
                         int baseline_max_it, double baseline_tol, int* ok, double* loc, double* width, double* bounds,
                         double* local_baseline, double* height, double* area, long long* idx_range);
int nmrfit_peaks_probe(nmrfit_peaks* h, int b, const long long* idx, int n, double* wu, double* uu, double* us);

/* Page-locked host memory for result buffers: device-to-host copies into it run at PCIe speed and skip the page
 * faults of freshly allocated pageable memory (generate_result at scale 16 writes 109 MB).  The Python layer pools these. */
int nmrfit_host_alloc(size_t bytes, void** out);
int nmrfit_host_free(void* p);

/* DFMA throughput of the device (TFLOP/s): best single launch and back-to-back average. */
int nmrfit_fp64_peak(int device, int iters, int repeats, double* burst_tflops, double* sustained_tflops);
/* Kernels launched by this library in this process since load (for bench.py's gpu_launches). */
long long nmrfit_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
