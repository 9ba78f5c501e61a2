// extern "C" surface of libnmrfit_b200.so (declared in include/nmrfit_b200.h).
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <utility>
#include <vector>
#include "../../include/nmrfit_b200.h"
#include "nmrfit_internal.h"

namespace nmrfit {
std::atomic<long long> g_launches{0};
void count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}

using namespace nmrfit;

namespace {

thread_local std::string t_error;

int fail(int code, const std::string& msg) {
    t_error = msg;
    return code;
}

int fail_cuda(cudaError_t e, const char* where) {
    t_error = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return NMRFIT_ERR_CUDA;
}

#define CK(call)                                              \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) return fail_cuda(_e, #call);   \
    } while (0)

// An array that grows on demand and is freed with its owner: device memory, or page-locked host memory.  The owner's
// device must be current when it is destroyed.
template <typename T, bool kPinned>
struct Buf {
    T* ptr = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : ptr(std::exchange(o.ptr, nullptr)), cap(std::exchange(o.cap, 0)) {}
    ~Buf() { release(); }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        release();
        cudaError_t e = kPinned ? cudaMallocHost((void**)&ptr, n * sizeof(T)) : cudaMalloc((void**)&ptr, n * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() {
        if (ptr && kPinned) cudaFreeHost(ptr);
        else if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
};
template <typename T> using DevBuf = Buf<T, false>;
template <typename T> using PinnedBuf = Buf<T, true>;

// One CUDA runtime object (stream, event, allocation, IPC mapping), destroyed with its owner
template <typename H, cudaError_t (*Destroy)(H)>
struct Owned {
    H h = nullptr;
    Owned() = default;
    explicit Owned(H v) : h(v) {}
    Owned(Owned&& o) noexcept : h(std::exchange(o.h, nullptr)) {}
    ~Owned() { if (h) Destroy(h); }
};
using Stream = Owned<cudaStream_t, cudaStreamDestroy>;
using Event = Owned<cudaEvent_t, cudaEventDestroy>;
using DevAlloc = Owned<void*, cudaFree>;
using IpcMapping = Owned<void*, cudaIpcCloseMemHandle>;

// the non-blocking stream of `s`, created on first use
cudaError_t ensure_stream(Stream& s) { return s.h ? cudaSuccess : cudaStreamCreateWithFlags(&s.h, cudaStreamNonBlocking); }

bool is_device_pointer(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

}  // namespace

constexpr int kShadowSpectra = 4;

struct nmrfit_ctx {
    int device = 0, B = 0, N = 0, P = 0, D = 0, precision = 0;
    DevBuf<double> spec;               // [B][4][N]
    std::vector<char> spec_set;
    std::vector<std::vector<double>> shadow;   // host copies of small contexts' spectra: an unchanged spectrum is not re-sent
    DevBuf<double> grid_h;             // [B][2] axis spacing h and 2^-52*max|w| of each spectrum
    std::vector<char> uniform;         // [B] stored w is w_0 + i*h to within 4 ulp
    int algorithm = NMRFIT_ALGO_AUTO;
    DevBuf<double> partials, x_stage, f_stage;
    DevBuf<double> prep_coef, prep_part, prep_far, prep_anchor;   // uniform-axis kernel, per-particle constants
    DevBuf<unsigned> prep_mask;
    ObjTune user_tune{0, 0, 0, 0, -1, 0, 0};   // variant -1, occ 0: the library's choice
    // swarm
    bool swarm = false;
    SwarmState sw{};
    int maxiter = 0, kk = 0, generation = 0;
    DevBuf<double> sx, sv, sp, sfx, sfp, sg, sfg, sbx, sbf, slb, sub, srec, rnd_a, rnd_b;
    DevBuf<int> sstop, sit;
    DevBuf<double> frec_f, frec_x;     // fused swarm kernel: published records
    DevBuf<unsigned> fbarrier;
    DevBuf<int> ferror;                // fused swarm kernel: barrier-timeout flag
    DevBuf<unsigned> mt_state;         // MT19937 key [624] + position, for nmrfit_ctx_mt19937
    DevBuf<unsigned> mt_words;         // ... and the tempered word stream of one call
    long long mt_elems = 0;            // elements of one random array (n_spectra * swarmsize * D)
    DevBuf<double> mt_a[2], mt_b[2];   // nmrfit_ctx_mt19937_begin / _end: two sets of arrays, used in turn
    DevBuf<unsigned> mt_state2, mt_words2;
    Stream mt_stream;
    PinnedBuf<unsigned> mt_host;       // [2][625]: state in, state out
    int mt_flip = 0, mt_pending = 0;
    DevBuf<double> fin_scratch;        // finish kernel: per-CTA candidates
    DevBuf<unsigned> fin_tickets;
    // record exchange over peer memory (particle sharding without a collective call)
    DevAlloc peer_win;                 // this context's window: records [2][R][B][D+2], then tokens [R][B]
    size_t peer_rec_bytes = 0;
    int peer_ranks = 0, peer_rank = 0;
    bool peers_ready = false;
    std::vector<IpcMapping> peer_opened;   // windows of other processes opened through CUDA IPC
    DevBuf<double*> peer_recs_dev;
    DevBuf<long long*> peer_tok_dev;
    DevBuf<int> peer_err;
    long long epoch = 0;               // fits begun on this context: part of the exchange token
    double peer_timeout_ms = 20000.0;  // wall-time bound of a wait for the peers' tokens
    DevBuf<double> wscratch, wbounds;  // batched weights: sweep scratch [B][N], windows + values
    DevBuf<double> ne_x, ne_part, ne_out;   // normal equations: positions, chunk partials, H | M | g | ssr
    DevBuf<double> lg_rho, lg_part, lg_out;   // lagged passes: rho, chunk partials, r or M_rho
    DevBuf<double> rf_x, rf_cur;       // refinement: current, trial, lb, ub [4][B][D]; H | g | s at the current point
    DevBuf<RefineState> rf_state;
    DevBuf<int> rf_active;             // spectra still running after the last polled step
    DevBuf<int> rf_tie_i;              // tied refinement: the tie map of each spectrum (RefineTies)
    DevBuf<double> rf_tie_d;
    DevBuf<double> rb_scale, rb_part, rb_out;   // robust losses: f_scale [B], moments chunk partials, moments [B][5]
    DevBuf<double> sc_res, sc_out;     // residual scale: residuals [B][N], (median, MAD) [B][2]
    Stream pipe[2];                    // nmrfit_objective_batch_host: slices of a large particle set
    PinnedBuf<double> h_f;             // ... and staging of their values
    int far_cells = 0;                 // far-field cells per region: 0 = far_cells_per_region(N, R), else 1 | 2 | 4
    int fused_mode = NMRFIT_FUSED_AUTO;
    DevBuf<long long> ftiming;         // optional per-phase cycle counters of the fused kernel
    bool fused_timing = false;
    long long fused_launches = 0;
    PinnedBuf<int> h_flags;            // [2*B]
    // optional per-launch timing of the objective kernel (nmrfit_ctx_profile)
    bool profiling = false;
    std::vector<Event> prof_events;    // triples
    size_t prof_used = 0;
};

struct nmrfit_phase {
    int device = 0, B = 0, N = 0;
    DevBuf<double> u, v, cands, out;   // spectra [B][N] x 2; candidates; err/score [B][K] + best [2][B]
    DevBuf<int> ok;
};

struct nmrfit_peaks {
    int device = 0, B = 0, N = 0, upsample = 100, max_peaks = 0;
    long long M = 0;
    int nblk = 0;
    DevBuf<double> w, u, uu, us, bmax, base, uu_at, pk_h, sg;
    DevBuf<long long> maxima, pk_i, cross, probe_idx;
    DevBuf<int> n_maxima, n_pk;
    DevBuf<char> out;
    DevBuf<double> probe_out;
    bool ran = false;
};

namespace {

// Is the axis uniform?  h = (w_last - w_0)/(N-1); every stored w_i within 4 ulp of w_0 + i*h.
// grid[0] = h, grid[1] = 2^-52 * max|w|.
bool axis_is_uniform(const double* hw, int N, double* grid) {
    double h = 0.0, big = 0.0;
    bool uni = N >= 2;
    if (uni) {
        h = (hw[N - 1] - hw[0]) / (double)(N - 1);
        big = std::max(std::fabs(hw[0]), std::fabs(hw[N - 1]));
        const double tol = 4.0 * 2.220446049250313e-16 * big;
        uni = std::isfinite(h) && h != 0.0 && std::isfinite(big);
        for (int i = 0; uni && i < N; ++i) uni = std::fabs(hw[i] - std::fma((double)i, h, hw[0])) <= tol;
    }
    grid[0] = h;
    grid[1] = 2.220446049250313e-16 * big;
    return uni;
}

// The launch plan of an objective call on this context (objective_plan.h)
ObjPlan ctx_plan(const nmrfit_ctx* c, int S, int fit_im, size_t slots_total = 0) {
    bool uniform_axis = true;
    for (char u : c->uniform) uniform_axis = uniform_axis && u;
    return objective_plan(c->N, c->P, S, c->B, c->precision, fit_im, uniform_axis, c->algorithm, c->user_tune,
                          c->far_cells, slots_total);
}

bool two_pass(const ObjPlan& p) { return p.kernel == OBJ_UNIFORM || p.kernel == OBJ_STREAM; }

int check_ctx(const nmrfit_ctx* c) {
    if (!c) return fail(NMRFIT_ERR_ARG, "ctx is NULL");
    return NMRFIT_OK;
}

// every spectrum of the context has been set; `what` completes the error message otherwise
int require_spectra(const nmrfit_ctx* c, const char* what) {
    for (char f : c->spec_set)
        if (!f) return fail(NMRFIT_ERR_STATE, std::string("every spectrum must be set before ") + what);
    return NMRFIT_OK;
}

// optional inputs of run_objective
struct ObjIn {
    const double* x_in = nullptr;      // the positions as the device sees them in page-locked host memory (FP64 uniform axis)
    // (one spectrum only) this launch is one slice of a larger particle set evaluated in pieces on several streams
    // (nmrfit_objective_batch_host); it owns the scratch of particle slots [slot0, slot0 + S + pad) of slots_total
    size_t slot0 = 0, slots_total = 0;
    const int* frozen = nullptr;       // per-spectrum stop flags of the swarm: stopped spectra are skipped
    const MoveArgs* move = nullptr;    // move the swarm before evaluating it
};

// what a launch of run_objective left in c->partials for the finish kernel
struct ObjOut {
    int n_tiles = 0, nsum = 1, nw = 1;
};

int run_objective(nmrfit_ctx* c, const double* x_dev, int S, int fit_im, double* f_dev, cudaStream_t st,
                  const ObjIn& in = {}, ObjOut* out = nullptr) {
    for (int b = 0; b < c->B; ++b)
        if (!c->spec_set[b]) return fail(NMRFIT_ERR_STATE, "spectrum " + std::to_string(b) + " was never set");
    if (fit_im < 0 || fit_im > 2) return fail(NMRFIT_ERR_ARG, "fit_im must be 0, 1 or 2");
    const ObjPlan p = ctx_plan(c, S, fit_im, in.slots_total);
    if (p.refuse) return fail(p.refuse, p.why);
    CK(c->partials.reserve(p.slots * p.part_per));
    ObjArgs a{};
    if (p.prep_threads) {
        const size_t slots = p.slots + p.pad;
        CK(c->prep_coef.reserve(slots * p.coef));
        CK(c->prep_part.reserve(slots * p.part));
        CK(c->prep_far.reserve(slots * p.far));
        CK(c->prep_anchor.reserve(slots * p.anchor));
        CK(c->prep_mask.reserve(slots * p.mask));
        a.prep_coef = c->prep_coef.ptr + in.slot0 * p.coef; a.prep_part = c->prep_part.ptr + in.slot0 * p.part;
        a.prep_far = c->prep_far.ptr + in.slot0 * p.far; a.prep_anchor = c->prep_anchor.ptr + in.slot0 * p.anchor;
        a.prep_mask = c->prep_mask.ptr + in.slot0 * p.mask;
    }
    a.spec = c->spec.ptr;
    a.x = x_dev;
    a.x_in = in.x_in;                                      // (two-pass FP64 path only: the caller checks)
    a.partials = c->partials.ptr + in.slot0 * p.part_per;
    a.frozen = in.frozen;
    a.grid_h = c->grid_h.ptr;
    a.N = c->N; a.P = c->P; a.S = S; a.kk = fit_im;
    // profiling: three events per launch - before the prepare pass, between it and the evaluation kernel, after
    cudaEvent_t ev[3] = {};
    if (c->profiling) {
        while (c->prof_events.size() < c->prof_used + 3) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            c->prof_events.emplace_back(e);
        }
        for (int k = 0; k < 3; ++k) ev[k] = c->prof_events[c->prof_used + k].h;
        c->prof_used += 3;
    }
    cudaError_t e = run_objective_plan(p, a, c->B, in.move, f_dev, st, ev[0], ev[1], ev[2]);
    if (e != cudaSuccess) return fail_cuda(e, "objective launch");
    if (out) *out = ObjOut{p.n_tiles, p.nsum, p.nw};
    return NMRFIT_OK;
}

// stage a [n] double array that may live on the host into `buf`; returns the device pointer to use
int stage(const double* src, size_t n, DevBuf<double>& buf, cudaStream_t st, const double** out) {
    if (!src) { *out = nullptr; return NMRFIT_OK; }
    if (is_device_pointer(src)) { *out = src; return NMRFIT_OK; }
    CK(buf.reserve(n));
    CK(cudaMemcpyAsync(buf.ptr, src, n * sizeof(double), cudaMemcpyHostToDevice, st));
    *out = buf.ptr;
    return NMRFIT_OK;
}

// The prologue of the post-fit entry points, in the order of their refusals: the context; `args`, the entry point's
// checks of its own arguments (NULL pointers first); at most 64 peaks (`peaks` opens that message); `plan_args`, its
// checks against the pass's plan; every spectrum set (`when` ends that message).  Then the device is made current and
// x [B][D] staged in *xd (x null stages nothing).
template <typename Args, typename PlanArgs>
int post_fit_begin(nmrfit_ctx* c, Args&& args, const char* peaks, PlanArgs&& plan_args, const char* when,
                   const double* x, cudaStream_t st, const double** xd) {
    if (int r = check_ctx(c)) return r;
    if (int r = args()) return r;
    if (c->P > 64)
        return fail(NMRFIT_ERR_ARG, std::string(peaks) + " at most 64 peaks (D <= 196), the context has " +
                                        std::to_string(c->P));
    if (int r = plan_args()) return r;
    if (int r = require_spectra(c, when)) return r;
    CK(cudaSetDevice(c->device));
    return stage(x, (size_t)c->B * c->D, c->ne_x, st, xd);
}

int no_checks() { return NMRFIT_OK; }

// Fill the fused kernel's arguments for `n_gen` generations and decide whether it can run (FP64, uniform axis,
// real-only fit, default exp table, and every CTA co-resident).
int fused_setup(nmrfit_ctx* c, int n_gen, const double* rp_d, const double* rg_d, FusedArgs* a, FusedPlan* plan) {
    plan->ok = false;
    if (c->fused_mode == NMRFIT_FUSED_OFF) return NMRFIT_OK;
    const SwarmState& s = c->sw;
    const ObjPlan p = ctx_plan(c, s.S, NMRFIT_REAL_ONLY);
    if (c->precision != NMRFIT_FP64 || c->kk != NMRFIT_REAL_ONLY || !two_pass(p)) return NMRFIT_OK;
    *a = FusedArgs{};
    a->s = s;
    a->spec = c->spec.ptr;
    a->grid_h = c->grid_h.ptr;
    a->rp = rp_d;
    a->rg = rg_d;
    a->N = c->N; a->P = c->P;
    a->n_vtiles = p.n_tiles;
    a->vw = p.t.threads / 32;
    a->sub = p.sub;
    a->n_gen = n_gen;
    a->gen0 = c->generation + 1;
    a->maxiter = c->maxiter;
    cudaError_t e = swarm_fused_plan(*a, c->D, s.B, s.S, p.t, c->device, c->fused_mode == NMRFIT_FUSED_REQUIRE, plan);
    if (e != cudaSuccess) return fail_cuda(e, "fused swarm plan");
    if (!plan->ok) return NMRFIT_OK;
    CK(c->frec_f.reserve(2 * (size_t)s.B * s.S));
    CK(c->frec_x.reserve(2 * (size_t)s.B * s.S * s.D));
    CK(c->fbarrier.reserve(s.B));
    if (!c->ferror.ptr) {
        CK(c->ferror.reserve(1));
        CK(cudaMemset(c->ferror.ptr, 0, sizeof(int)));
    }
    a->error = c->ferror.ptr;
    a->max_wait_ns = 10LL * 1000 * 1000 * 1000;            // 10 s; the legitimate wait is microseconds
    a->rec_f = c->frec_f.ptr;
    a->rec_x = c->frec_x.ptr;
    a->barrier = c->fbarrier.ptr;
    a->timing = c->fused_timing ? c->ftiming.ptr : nullptr;
    return NMRFIT_OK;
}

// One generation of the per-step path in three launches: [move + per-particle constants], [objective tiles],
// [tile sums + personal bests + local best record (+ swarm-best commit)].  generation 0 (`move` false) evaluates
// the freshly initialised swarm.
PeerArgs make_peer_args(const nmrfit_ctx* c) {
    PeerArgs pa{};
    pa.recs = c->peer_recs_dev.ptr;
    pa.tokens = c->peer_tok_dev.ptr;
    pa.n_ranks = c->peer_ranks;
    pa.rank = c->peer_rank;
    pa.token = (c->epoch << 32) | (long long)c->generation;
    pa.max_wait_ns = (long long)(c->peer_timeout_ms * 1e6);
    pa.error = c->peer_err.ptr;
    return pa;
}

// commit: 0 none (the caller exchanges the records itself), 1 this context's own record, 2 the ranks' records
// exchanged over peer memory inside the finish kernel
int swarm_generation(nmrfit_ctx* c, bool move, const double* rp_d, const double* rg_d, int commit, cudaStream_t st) {
    SwarmState& s = c->sw;
    if (commit == 2 && !c->peers_ready) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_peer_open has not been called");
    const PeerArgs pa = commit == 2 ? make_peer_args(c) : PeerArgs{};
    const MoveArgs mv{s, rp_d, rg_d, c->generation};
    ObjIn in;
    if (move) {
        in.frozen = s.stop;
        in.move = &mv;
    }
    ObjOut o;
    if (int rc = run_objective(c, s.x, s.S, c->kk, nullptr, st, in, &o)) return rc;
    cudaError_t e = launch_swarm_finish(s, c->partials.ptr, o.n_tiles, o.nsum, c->N, s.rec, c->fin_scratch.ptr,
                                        c->fin_tickets.ptr, commit, c->maxiter, st, o.nw, commit == 2 ? &pa : nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "swarm finish");
    return NMRFIT_OK;
}

int require_swarm(const nmrfit_ctx* c) {
    if (int rc = check_ctx(c)) return rc;
    if (!c->swarm) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_begin has not been called");
    return NMRFIT_OK;
}

// The random arrays of `n` generations, [n][B][S][D] each: both given (host arrays are staged into rnd_a / rnd_b,
// device arrays are used in place) or both null (the swarm draws its own).  `names` is how the caller calls them.
int stage_random(nmrfit_ctx* c, int n, const double* rp, const double* rg, const char* names, cudaStream_t st,
                 const double** rp_d, const double** rg_d) {
    *rp_d = *rg_d = nullptr;
    if ((rp == nullptr) != (rg == nullptr)) return fail(NMRFIT_ERR_ARG, std::string(names) + " must both be given or both be NULL");
    if (n <= 0) return NMRFIT_OK;
    const size_t nsd = (size_t)c->sw.B * c->sw.S * c->sw.D * n;
    if (int rc = stage(rp, nsd, c->rnd_a, st, rp_d)) return rc;
    return stage(rg, nsd, c->rnd_b, st, rg_d);
}

// `n` generations of the per-step path on `st`, with the random arrays of stage_random
int queue_generations(nmrfit_ctx* c, int n, const double* rp_d, const double* rg_d, int commit, cudaStream_t st) {
    const size_t nsd = (size_t)c->sw.B * c->sw.S * c->sw.D;
    for (int k = 0; k < n; ++k) {
        c->generation += 1;
        if (int rc = swarm_generation(c, true, rp_d ? rp_d + nsd * k : nullptr, rg_d ? rg_d + nsd * k : nullptr, commit, st))
            return rc;
    }
    return NMRFIT_OK;
}

// Queue the host copy of the stop flags into h_flags [0, B) and of an optional device error word into h_flags [B] (0
// without one).  Once `st` has been synchronised, running_spectra counts the spectra whose swarm has not stopped.
int queue_stop_flags(nmrfit_ctx* c, const int* err_dev, cudaStream_t st) {
    const int B = c->sw.B;
    CK(cudaMemcpyAsync(c->h_flags.ptr, c->sw.stop, sizeof(int) * B, cudaMemcpyDeviceToHost, st));
    c->h_flags.ptr[B] = 0;
    if (err_dev) CK(cudaMemcpyAsync(c->h_flags.ptr + B, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    return NMRFIT_OK;
}

int running_spectra(const nmrfit_ctx* c) {
    int running = 0;
    for (int b = 0; b < c->sw.B; ++b) running += c->h_flags.ptr[b] == 0;
    return running;
}

}  // namespace

extern "C" {

int nmrfit_abi_version(void) { return NMRFIT_ABI_VERSION; }

const char* nmrfit_last_error(void) { return t_error.c_str(); }

int nmrfit_device_count(int* count) {
    if (!count) return fail(NMRFIT_ERR_ARG, "count is NULL");
    CK(cudaGetDeviceCount(count));
    return NMRFIT_OK;
}

long long nmrfit_launch_count(void) { return g_launches.load(); }

int nmrfit_ctx_create(nmrfit_ctx** out, int device, int n_spectra, int n_points, int n_peaks, int precision) {
    if (!out) return fail(NMRFIT_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (n_spectra < 1 || n_points < 1 || n_peaks < 1) return fail(NMRFIT_ERR_ARG, "n_spectra, n_points, n_peaks must be >= 1");
    if (n_peaks > 256) return fail(NMRFIT_ERR_ARG, "n_peaks > 256 is not supported");
    if (precision != NMRFIT_FP64 && precision != NMRFIT_FP32) return fail(NMRFIT_ERR_ARG, "unknown precision");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(NMRFIT_ERR_ARG, "no such CUDA device");
    CK(cudaSetDevice(device));
    std::unique_ptr<nmrfit_ctx> c(new (std::nothrow) nmrfit_ctx());
    if (!c) return fail(NMRFIT_ERR_NOMEM, "out of host memory");
    c->device = device; c->B = n_spectra; c->N = n_points; c->P = n_peaks; c->D = 4 + 3 * n_peaks;
    c->precision = precision;
    c->spec_set.assign(n_spectra, 0);
    c->uniform.assign(n_spectra, 0);
    CK(c->spec.reserve((size_t)n_spectra * 4 * n_points));
    CK(c->grid_h.reserve(2 * (size_t)n_spectra));
    CK(c->h_flags.reserve(2 * (size_t)n_spectra));
    *out = c.release();
    return NMRFIT_OK;
}

void nmrfit_ctx_destroy(nmrfit_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    delete c;
}

int nmrfit_ctx_set_spectrum(nmrfit_ctx* c, int b, const double* w, const double* u, const double* v,
                            const double* weights) {
    if (int r = check_ctx(c)) return r;
    if (b < 0 || b >= c->B) return fail(NMRFIT_ERR_ARG, "spectrum index out of range");
    if (!w || !u || !v || !weights) return fail(NMRFIT_ERR_ARG, "w, u, v, weights must be non-NULL");
    CK(cudaSetDevice(c->device));
    double* dst = c->spec.ptr + (size_t)b * 4 * c->N;
    const double* src[4] = {w, u, v, weights};
    // Callers that keep the reference's calling convention (objective(x, w, u, v, weights) per call) hand over the
    // same spectrum again and again: contexts of up to kShadowSpectra spectra keep a host copy and skip the upload
    // and the axis check when the four arrays are byte-identical to what the device already holds.
    const bool host_src = !is_device_pointer(w) && !is_device_pointer(u) && !is_device_pointer(v) && !is_device_pointer(weights);
    const bool shadowed = c->B <= kShadowSpectra && host_src;
    const size_t plane = sizeof(double) * (size_t)c->N;
    if (shadowed) {
        if (c->shadow.empty()) c->shadow.resize(c->B);
        std::vector<double>& sh = c->shadow[b];
        if (c->spec_set[b] && sh.size() == 4 * (size_t)c->N) {
            bool same = true;
            for (int k = 0; same && k < 4; ++k) same = std::memcmp(sh.data() + (size_t)k * c->N, src[k], plane) == 0;
            if (same) return NMRFIT_OK;
        }
        sh.resize(4 * (size_t)c->N);
        for (int k = 0; k < 4; ++k) std::memcpy(sh.data() + (size_t)k * c->N, src[k], plane);
    } else if (!c->shadow.empty()) {
        c->shadow[b].clear();
    }
    for (int k = 0; k < 4; ++k)
        CK(cudaMemcpy(dst + (size_t)k * c->N, src[k], sizeof(double) * c->N, cudaMemcpyDefault));
    std::vector<double> hw;
    const double* wh = w;                                  // checked on the host: the caller's memory if it is host memory
    if (is_device_pointer(w)) {
        hw.resize(c->N);
        CK(cudaMemcpy(hw.data(), dst, sizeof(double) * c->N, cudaMemcpyDeviceToHost));
        wh = hw.data();
    }
    double grid[2];
    c->uniform[b] = axis_is_uniform(wh, c->N, grid) ? 1 : 0;
    CK(cudaMemcpy(c->grid_h.ptr + 2 * (size_t)b, grid, sizeof(grid), cudaMemcpyHostToDevice));
    c->spec_set[b] = 1;
    return NMRFIT_OK;
}

int nmrfit_ctx_set_spectra(nmrfit_ctx* c, int b0, int count, const double* w, const double* u, const double* v,
                           const double* weights) {
    if (int r = check_ctx(c)) return r;
    if (b0 < 0 || count < 1 || b0 + count > c->B) return fail(NMRFIT_ERR_ARG, "spectrum range out of bounds");
    if (!w || !u || !v) return fail(NMRFIT_ERR_ARG, "w, u, v must be non-NULL");
    CK(cudaSetDevice(c->device));
    for (auto& sh : c->shadow) sh.clear();                 // the device copy changes behind the shadows
    const size_t N = (size_t)c->N, row = sizeof(double) * N;
    double* dst = c->spec.ptr + (size_t)b0 * 4 * N;
    const double* src[4] = {w, u, v, weights};
    for (int k = 0; k < 4; ++k) {
        if (!src[k]) continue;                             // weights may follow from nmrfit_ctx_compute_weights
        CK(cudaMemcpy2D(dst + k * N, 4 * row, src[k], row, row, count, cudaMemcpyDefault));
    }
    // uniformity of every axis, on the host: straight from the caller's memory when that is host memory
    std::vector<double> hw;
    const double* wh = w;
    if (is_device_pointer(w)) {
        hw.resize((size_t)count * N);
        CK(cudaMemcpy(hw.data(), w, row * count, cudaMemcpyDeviceToHost));
        wh = hw.data();
    }
    std::vector<double> grid(2 * (size_t)count);
    for (int i = 0; i < count; ++i) {
        c->uniform[b0 + i] = axis_is_uniform(wh + (size_t)i * N, c->N, &grid[2 * (size_t)i]) ? 1 : 0;
        c->spec_set[b0 + i] = 1;
    }
    CK(cudaMemcpy(c->grid_h.ptr + 2 * (size_t)b0, grid.data(), sizeof(double) * grid.size(), cudaMemcpyHostToDevice));
    return NMRFIT_OK;
}

int nmrfit_ctx_compute_weights(nmrfit_ctx* c, const double* peak_bounds, const double* peak_values, int n_windows,
                               int sweeps, double omega, double* weights_out, void* stream) {
    if (int r = check_ctx(c)) return r;
    if (!peak_bounds || !peak_values) return fail(NMRFIT_ERR_ARG, "peak_bounds and peak_values must be non-NULL");
    if (n_windows < 1 || n_windows > 4096) return fail(NMRFIT_ERR_ARG, "n_windows must be 1..4096");
    if (sweeps < 0) return fail(NMRFIT_ERR_ARG, "sweeps must be >= 0");
    if (int r = require_spectra(c, "its weights are computed")) return r;
    CK(cudaSetDevice(c->device));
    for (auto& sh : c->shadow) sh.clear();                 // the weights plane is rewritten on the device
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)c->B, N = (size_t)c->N, nb = B * 2 * n_windows, nv = B * n_windows;
    CK(c->wscratch.reserve(B * N));
    CK(c->wbounds.reserve(nb + nv));
    CK(cudaMemcpyAsync(c->wbounds.ptr, peak_bounds, sizeof(double) * nb, cudaMemcpyDefault, st));
    CK(cudaMemcpyAsync(c->wbounds.ptr + nb, peak_values, sizeof(double) * nv, cudaMemcpyDefault, st));
    cudaError_t e = launch_weights(c->spec.ptr, c->wscratch.ptr, c->wbounds.ptr, c->wbounds.ptr + nb, c->B, c->N,
                                   n_windows, sweeps, omega, st);
    if (e != cudaSuccess) return fail_cuda(e, "weights launch");
    if (weights_out)
        CK(cudaMemcpy2DAsync(weights_out, sizeof(double) * N, c->spec.ptr + 3 * N, sizeof(double) * 4 * N,
                             sizeof(double) * N, B, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // the staged bounds may be pageable host memory
    return NMRFIT_OK;
}

static int check_loss(int loss) {
    if (loss < NMRFIT_LOSS_LINEAR || loss > NMRFIT_LOSS_CAUCHY)
        return fail(NMRFIT_ERR_ARG, "unknown loss " + std::to_string(loss) + " (NMRFIT_LOSS_LINEAR, _HUBER, _SOFT_L1 "
                                    "or _CAUCHY)");
    return NMRFIT_OK;
}

// A robust loss's f_scale [B] (host or device) read, checked and staged on the device in *dev.  *dev stays null for
// LINEAR, whose f_scale is not read.
static int stage_loss(nmrfit_ctx* c, int loss, const double* f_scale, cudaStream_t st, const double** dev) {
    *dev = nullptr;
    if (loss == NMRFIT_LOSS_LINEAR) return NMRFIT_OK;
    if (!f_scale) return fail(NMRFIT_ERR_ARG, "f_scale must be non-NULL for a robust loss");
    std::vector<double> h(c->B);
    CK(cudaMemcpy(h.data(), f_scale, sizeof(double) * c->B, cudaMemcpyDefault));
    for (int b = 0; b < c->B; ++b)
        if (!(std::isfinite(h[b]) && h[b] > 0.0))
            return fail(NMRFIT_ERR_ARG, "spectrum " + std::to_string(b) + ": f_scale must be finite and > 0");
    CK(c->rb_scale.reserve(c->B));
    CK(cudaMemcpyAsync(c->rb_scale.ptr, h.data(), sizeof(double) * c->B, cudaMemcpyHostToDevice, st));
    *dev = c->rb_scale.ptr;
    return NMRFIT_OK;
}

// Both normal-equations entry points: the pass of `loss` (launch_normal_eq_loss, LINEAR is K12), then the blocks
// dst[k] that are non-null copied out of each spectrum's H [D][D] | M [D][D] | g [D] | ssr [2], n_ssr entries of ssr.
// `pass` names the pass in the messages.
static int normal_eq_pass(nmrfit_ctx* c, const double* x, int loss, const double* f_scale, const char* pass,
                          const char* when, double* const dst[4], size_t n_ssr, cudaStream_t st) {
    const double* xd = nullptr;
    if (int r = post_fit_begin(
            c, [&] { return x ? check_loss(loss) : fail(NMRFIT_ERR_ARG, "x must be non-NULL"); },
            (std::string(pass) + " support").c_str(), no_checks, when, x, st, &xd))
        return r;
    const double* fs = nullptr;
    if (int r = stage_loss(c, loss, f_scale, st, &fs)) return r;
    const size_t B = (size_t)c->B, D = (size_t)c->D, DD = D * D, per = 2 * DD + D + 2;
    const NormalEqPlan p = normal_eq_plan(c->N, c->P);
    CK(c->ne_part.reserve(normal_eq_scratch_doubles(p, c->B)));
    CK(c->ne_out.reserve(B * per));
    cudaError_t e = launch_normal_eq_loss(c->spec.ptr, xd, loss, fs, p, c->B, c->ne_part.ptr, c->ne_out.ptr, st);
    if (e != cudaSuccess) return fail_cuda(e, (std::string(pass) + " launch").c_str());
    const size_t offs[4] = {0, DD, 2 * DD, 2 * DD + D}, lens[4] = {DD, DD, D, n_ssr};
    for (int k = 0; k < 4; ++k)
        if (dst[k])
            CK(cudaMemcpy2DAsync(dst[k], sizeof(double) * lens[k], c->ne_out.ptr + offs[k], sizeof(double) * per,
                                 sizeof(double) * lens[k], B, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // x and the outputs may be pageable host memory
    return NMRFIT_OK;
}

int nmrfit_ctx_normal_equations(nmrfit_ctx* c, const double* x, double* H, double* M, double* g, double* ssr,
                                void* stream) {
    double* const dst[4] = {H, M, g, ssr};
    return normal_eq_pass(c, x, NMRFIT_LOSS_LINEAR, nullptr, "normal equations", "its normal equations are computed",
                          dst, 2, (cudaStream_t)stream);
}

// the robust pass's block is H_rho | M | g_rho | (cost, sum w^2 rho' res^2): H, g and the cost are copied out
int nmrfit_ctx_normal_equations_loss(nmrfit_ctx* c, const double* x, int loss, const double* f_scale, double* H,
                                     double* g, double* cost, void* stream) {
    double* const dst[4] = {H, nullptr, g, cost};
    return normal_eq_pass(c, x, loss, f_scale, "robust normal equations", "a robust pass runs", dst, 1,
                          (cudaStream_t)stream);
}

int nmrfit_ctx_loss_moments(nmrfit_ctx* c, const double* x, int loss, const double* f_scale, double* out,
                            void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const double* xd = nullptr;
    if (int r = post_fit_begin(
            c, [&] { return x && out ? check_loss(loss) : fail(NMRFIT_ERR_ARG, "x and out must be non-NULL"); },
            "loss moments support", no_checks, "a robust pass runs", x, st, &xd))
        return r;
    const double* fs = nullptr;
    if (int r = stage_loss(c, loss, f_scale, st, &fs)) return r;
    const size_t B = (size_t)c->B;
    CK(c->rb_part.reserve(loss_moments_scratch_doubles(c->B, c->N)));
    CK(c->rb_out.reserve(B * 5));
    cudaError_t e = launch_loss_moments(c->spec.ptr, xd, loss, fs, c->B, c->N, c->P, c->rb_part.ptr, c->rb_out.ptr, st);
    if (e != cudaSuccess) return fail_cuda(e, "loss moments launch");
    CK(cudaMemcpyAsync(out, c->rb_out.ptr, sizeof(double) * B * 5, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // x and out may be pageable host memory
    return NMRFIT_OK;
}

// Both residual-scale entry points (DESIGN K17): the residuals at x into sc_res, then with `scale` their median and
// MAD into sc_out; `out` receives whichever was asked for.
static int residual_scale_pass(nmrfit_ctx* c, const double* x, bool scale, double* out, cudaStream_t st) {
    const double* xd = nullptr;
    if (int r = post_fit_begin(
            c, [&] { return x && out ? NMRFIT_OK : fail(NMRFIT_ERR_ARG, "x and out must be non-NULL"); },
            "the residual passes support", no_checks, "its residuals are computed", x, st, &xd))
        return r;
    const size_t B = (size_t)c->B, N = (size_t)c->N;
    CK(c->sc_res.reserve(B * N));
    cudaError_t e = launch_residuals(c->spec.ptr, xd, c->B, c->N, c->P, c->sc_res.ptr, st);
    if (e != cudaSuccess) return fail_cuda(e, "residuals launch");
    if (scale) {
        CK(c->sc_out.reserve(B * 2));
        e = launch_median_mad(c->sc_res.ptr, c->B, c->N, c->sc_out.ptr, st);
        if (e != cudaSuccess) return fail_cuda(e, "median and MAD launch");
        CK(cudaMemcpyAsync(out, c->sc_out.ptr, sizeof(double) * B * 2, cudaMemcpyDefault, st));
    } else {
        CK(cudaMemcpyAsync(out, c->sc_res.ptr, sizeof(double) * B * N, cudaMemcpyDefault, st));
    }
    CK(cudaStreamSynchronize(st));                         // x and out may be pageable host memory
    return NMRFIT_OK;
}

int nmrfit_ctx_residuals(nmrfit_ctx* c, const double* x, double* res_out, void* stream) {
    return residual_scale_pass(c, x, false, res_out, (cudaStream_t)stream);
}

int nmrfit_ctx_residual_scale(nmrfit_ctx* c, const double* x, double* out, void* stream) {
    return residual_scale_pass(c, x, true, out, (cudaStream_t)stream);
}

// the lag checks of both lagged passes; fills the plan
static int lagged_check(const nmrfit_ctx* c, int max_lag, LaggedPlan* plan) {
    if (max_lag < 0) return fail(NMRFIT_ERR_ARG, "max_lag must be >= 0");
    if (max_lag >= c->N)
        return fail(NMRFIT_ERR_ARG, "max_lag must be below the number of points, " + std::to_string(c->N));
    *plan = lagged_plan(c->N, c->P, max_lag);
    if (max_lag > plan->max_lag)
        return fail(NMRFIT_ERR_ARG, "max_lag " + std::to_string(max_lag) + " is above the cap of " +
                                        std::to_string(plan->max_lag) + " at " + std::to_string(c->P) + " peaks");
    return NMRFIT_OK;
}

int nmrfit_ctx_residual_acf(nmrfit_ctx* c, const double* x, int max_lag, double* r_out, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    LaggedPlan p;
    const double* xd = nullptr;
    if (int r = post_fit_begin(
            c, [&] { return x && r_out ? NMRFIT_OK : fail(NMRFIT_ERR_ARG, "x and r_out must be non-NULL"); },
            "the lagged passes support", [&] { return lagged_check(c, max_lag, &p); },
            "its residual autocorrelation is computed", x, st, &xd))
        return r;
    const size_t B = (size_t)c->B, K = (size_t)max_lag + 1;
    CK(c->lg_part.reserve(residual_acf_scratch_doubles(p, c->B)));
    CK(c->lg_out.reserve(B * K));
    cudaError_t e = launch_residual_acf(c->spec.ptr, xd, p, c->B, c->lg_part.ptr, c->lg_out.ptr, st);
    if (e != cudaSuccess) return fail_cuda(e, "residual autocorrelation launch");
    CK(cudaMemcpyAsync(r_out, c->lg_out.ptr, sizeof(double) * B * K, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // x and r_out may be pageable host memory
    return NMRFIT_OK;
}

int nmrfit_ctx_normal_m_lagged(nmrfit_ctx* c, const double* x, const double* rho, int max_lag, double* M_out,
                               void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    LaggedPlan p;
    std::vector<double> h;
    // rho is read and checked before the spectra are: it may be device memory, so with the device current
    auto rho_check = [&] {
        if (int r = lagged_check(c, max_lag, &p)) return r;
        CK(cudaSetDevice(c->device));
        h.resize((size_t)c->B * (max_lag + 1));
        CK(cudaMemcpy(h.data(), rho, sizeof(double) * h.size(), cudaMemcpyDefault));
        for (double v : h)
            if (!std::isfinite(v)) return fail(NMRFIT_ERR_ARG, "every rho must be finite");
        return NMRFIT_OK;
    };
    auto args = [&] {
        return x && rho && M_out ? NMRFIT_OK : fail(NMRFIT_ERR_ARG, "x, rho and M_out must be non-NULL");
    };
    const double* xd = nullptr;
    if (int r = post_fit_begin(c, args, "the lagged passes support", rho_check, "its lagged M is computed", x, st, &xd))
        return r;
    const size_t B = (size_t)c->B, D = (size_t)c->D;
    CK(c->lg_rho.reserve(h.size()));
    CK(cudaMemcpyAsync(c->lg_rho.ptr, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice, st));
    CK(c->lg_part.reserve(lagged_m_scratch_doubles(p, c->B)));
    CK(c->lg_out.reserve(B * D * D));
    cudaError_t e = launch_lagged_m(c->spec.ptr, xd, c->lg_rho.ptr, p, c->B, c->lg_part.ptr, c->lg_out.ptr, st);
    if (e != cudaSuccess) return fail_cuda(e, "lagged M launch");
    CK(cudaMemcpyAsync(M_out, c->lg_out.ptr, sizeof(double) * B * D * D, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // x, rho and M_out may be pageable host memory
    return NMRFIT_OK;
}

int nmrfit_lagged_plan(int n_points, int n_peaks, int max_lag, int* out) {
    if (!out) return fail(NMRFIT_ERR_ARG, "out is NULL");
    if (n_peaks < 1 || n_peaks > 64) return fail(NMRFIT_ERR_ARG, "n_peaks must be 1..64");
    if (n_points < 1) return fail(NMRFIT_ERR_ARG, "n_points must be >= 1");
    if (max_lag < 0) return fail(NMRFIT_ERR_ARG, "max_lag must be >= 0");
    const LaggedPlan p = lagged_plan(n_points, n_peaks, max_lag);
    if (max_lag > p.max_lag)
        return fail(NMRFIT_ERR_ARG, "max_lag " + std::to_string(max_lag) + " is above the cap of " +
                                        std::to_string(p.max_lag) + " at " + std::to_string(n_peaks) + " peaks");
    const int v[14] = {p.ng, p.slices, p.tasks, p.tasks_per_slice, p.threads, p.tp, p.chunk, p.n_chunks, (int)p.smem,
                       (int)lagged_m_scratch_doubles(p, 1), p.max_lag, p.acf_chunk, p.acf_n_chunks,
                       (int)residual_acf_scratch_doubles(p, 1)};
    for (int k = 0; k < 14; ++k) out[k] = v[k];
    return NMRFIT_OK;
}

constexpr int kRefinePoll = 8;   // refinement iterations queued between host reads of the running count

// the refinement's checks past the peak count
// (the tied refinement needs more points than free parameters only: build_ties checks that)
static int refine_check(const nmrfit_ctx* c, int max_iter, double xtol, bool tied) {
    if (!tied && c->N <= c->D) return fail(NMRFIT_ERR_ARG, "refinement needs more points than parameters");
    if (max_iter < 1) return fail(NMRFIT_ERR_ARG, "max_iter must be >= 1");
    if (!(xtol > 0.0)) return fail(NMRFIT_ERR_ARG, "xtol must be > 0");
    return NMRFIT_OK;
}

// The refinement loop of both entry points: h = [x | x | lb | ub] (the start is the first current point and the first
// trial; for tied parameters lb, ub hold the reduced box), ties null or on the device.
// `loss` and `fscale` (on the device, null for LINEAR) choose the pass (launch_normal_eq_loss).
static int refine_run(nmrfit_ctx* c, const std::vector<double>& h, const RefineTies* ties, int loss,
                      const double* fscale, int max_iter, double xtol, double* x, double* f_out, int* passes_out,
                      int* accepted_out, int* status_out, cudaStream_t st) {
    const size_t B = (size_t)c->B, D = (size_t)c->D, BD = B * D;
    const NormalEqPlan p = normal_eq_plan(c->N, c->P);
    CK(c->ne_part.reserve(normal_eq_scratch_doubles(p, c->B)));
    CK(c->ne_out.reserve(B * (2 * D * D + D + 2)));
    CK(c->rf_x.reserve(4 * BD));
    CK(c->rf_cur.reserve(B * (D * D + D + 1)));
    CK(c->rf_state.reserve(B));
    CK(c->rf_active.reserve(1));
    double *xc = c->rf_x.ptr, *xt = xc + BD, *lbd = xc + 2 * BD, *ubd = xc + 3 * BD;
    CK(cudaMemcpyAsync(xc, h.data(), sizeof(double) * 4 * BD, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(c->rf_state.ptr, 0, sizeof(RefineState) * B, st));
    // every running spectrum has had the same number of passes, so max_iter iterations finish them all
    for (int it = 0; it < max_iter; ++it) {
        cudaError_t e = launch_normal_eq_loss(c->spec.ptr, xt, loss, fscale, p, c->B, c->ne_part.ptr, c->ne_out.ptr, st);
        if (e != cudaSuccess) return fail_cuda(e, "refinement: normal equations launch");
        const bool poll = (it + 1) % kRefinePoll == 0 && it + 1 < max_iter;
        if (poll) CK(cudaMemsetAsync(c->rf_active.ptr, 0, sizeof(int), st));
        e = launch_refine_step(c->ne_out.ptr, c->rf_cur.ptr, c->rf_state.ptr, xc, xt, lbd, ubd, c->B, c->N, c->D,
                               max_iter, xtol, poll ? c->rf_active.ptr : nullptr, ties, st);
        if (e != cudaSuccess) return fail_cuda(e, "refinement step launch");
        if (poll) {
            CK(cudaMemcpyAsync(c->h_flags.ptr, c->rf_active.ptr, sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (c->h_flags.ptr[0] == 0) break;
        }
    }
    CK(cudaMemcpyAsync(x, xc, sizeof(double) * BD, cudaMemcpyDefault, st));
    const RefineState* rs = c->rf_state.ptr;
    const size_t pitch = sizeof(RefineState);
    if (f_out) CK(cudaMemcpy2DAsync(f_out, sizeof(double), &rs->f, pitch, sizeof(double), B, cudaMemcpyDefault, st));
    int* outs[3] = {passes_out, accepted_out, status_out};
    const int* srcs[3] = {&rs->passes, &rs->accepted, &rs->status};
    for (int k = 0; k < 3; ++k)
        if (outs[k]) CK(cudaMemcpy2DAsync(outs[k], sizeof(int), srcs[k], pitch, sizeof(int), B, cudaMemcpyDefault, st));
    CK(cudaStreamSynchronize(st));                         // the staged starts and the outputs may be pageable memory
    return NMRFIT_OK;
}

// the untied refinement past the prologue of nmrfit_ctx_refine_loss
static int refine_untied(nmrfit_ctx* c, double* x, const double* lb, const double* ub, int loss, const double* fscale,
                         int max_iter, double xtol, double* f_out, int* passes_out, int* accepted_out, int* status_out,
                         cudaStream_t st) {
    const size_t BD = (size_t)c->B * c->D;
    std::vector<double> h(4 * BD);
    CK(cudaMemcpy(h.data(), x, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(h.data() + 2 * BD, lb, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(h.data() + 3 * BD, ub, sizeof(double) * BD, cudaMemcpyDefault));
    std::copy(h.begin(), h.begin() + BD, h.begin() + BD);
    for (size_t i = 0; i < BD; ++i) {
        const double xi = h[i], lo = h[2 * BD + i], hi = h[3 * BD + i];
        if (!(hi > lo)) return fail(NMRFIT_ERR_ARG, "every lower bound must be below its upper bound");
        if (!(xi >= lo && xi <= hi)) return fail(NMRFIT_ERR_ARG, "the start must lie inside its box");
    }
    return refine_run(c, h, nullptr, loss, fscale, max_iter, xtol, x, f_out, passes_out, accepted_out, status_out, st);
}

// One spectrum's tie map checked, with its start and box, and turned into the kernel's layout: ti [3D + 2] and
// td [2D] (RefineTies), the reduced box in lo, hi [D] (first d entries), the start expanded in place in x [D].
static int build_ties(int b, int D, int N, const int* master, const double* scale, const double* offset, double* x,
                      const double* lb, const double* ub, int* ti, double* td, double* lo, double* hi) {
    const std::string at = "spectrum " + std::to_string(b) + ", parameter ";
    for (int j = 0; j < D; ++j) {
        const int m = master[j];
        if (m < -1 || m >= D)
            return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + ": master " + std::to_string(m) +
                                            " is out of range (-1 fixed, j free, else a free parameter below " +
                                            std::to_string(D) + ")");
        if (m == j) continue;
        if (!std::isfinite(offset[j])) return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + ": offset is not finite");
        if (m == -1) continue;
        if (!std::isfinite(scale[j]) || scale[j] == 0.0)
            return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + ": scale must be finite and non-zero (fix the "
                                            "parameter instead of a zero scale)");
        if (master[m] == -1)
            return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + ": its master " + std::to_string(m) + " is fixed");
        if (master[m] != m)
            return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + ": its master " + std::to_string(m) +
                                            " is itself linked (no chains)");
    }
    int* off = ti + 1;
    int* mem = ti + D + 2;
    int* fm = ti + 2 * D + 2;
    double* a = td;
    double* c = td + D;
    int d = 0, k = 0;
    for (int j = 0; j < D; ++j) {
        if (master[j] != j) continue;
        // the reduced box of theta_d: the master's own box intersected with each dependent's, mapped through it
        double l = lb[j], u = ub[j];
        if (!(u > l))
            return fail(NMRFIT_ERR_ARG, at + std::to_string(j) + " (a master or free): its box is empty or a single "
                                            "point");
        off[d] = k;
        fm[d] = j;
        for (int i = 0; i < D; ++i) {
            if (i != j && master[i] != j) continue;
            mem[k] = i;
            a[k] = i == j ? 1.0 : scale[i];
            c[k] = i == j ? 0.0 : offset[i];
            ++k;
            if (i == j) continue;
            double li = (lb[i] - offset[i]) / scale[i], ui = (ub[i] - offset[i]) / scale[i];
            if (scale[i] < 0.0) std::swap(li, ui);
            l = std::max(l, li);
            u = std::min(u, ui);
            if (!(u > l) || std::isnan(li) || std::isnan(ui))
                return fail(NMRFIT_ERR_ARG, at + std::to_string(i) + " and its master " + std::to_string(j) +
                                                ": the reduced box is empty or a single point");
        }
        lo[d] = l;
        hi[d] = u;
        x[j] = std::fmin(std::fmax(x[j], l), u);
        ++d;
    }
    off[d] = k;
    ti[0] = d;
    if (N <= d)
        return fail(NMRFIT_ERR_ARG, "spectrum " + std::to_string(b) + ": refinement needs more points than free "
                                    "parameters");
    for (int m = 0; m < d; ++m)                            // the expansion, as the step kernel makes it (no FMA)
        for (int q = off[m]; q < off[m + 1]; ++q)
            if (mem[q] != fm[m]) {
                volatile double t = a[q] * x[fm[m]];
                x[mem[q]] = t + c[q];
            }
    for (int j = 0; j < D; ++j)
        if (master[j] == -1) x[j] = offset[j];
    return NMRFIT_OK;
}

// the tied refinement past the prologue of nmrfit_ctx_refine_loss
static int refine_tied(nmrfit_ctx* c, double* x, const double* lb, const double* ub, const int* tie_master,
                       const double* tie_scale, const double* tie_offset, int loss, const double* fscale, int max_iter,
                       double xtol, double* f_out, int* passes_out, int* accepted_out, int* status_out,
                       cudaStream_t st) {
    const size_t B = (size_t)c->B, D = (size_t)c->D, BD = B * D;
    std::vector<double> h(4 * BD, 0.0), box(2 * BD), sc(BD), of(BD), td(2 * BD, 0.0);
    std::vector<int> ms(BD), ti(B * (3 * D + 2), 0);
    CK(cudaMemcpy(h.data(), x, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(box.data(), lb, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(box.data() + BD, ub, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(ms.data(), tie_master, sizeof(int) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(sc.data(), tie_scale, sizeof(double) * BD, cudaMemcpyDefault));
    CK(cudaMemcpy(of.data(), tie_offset, sizeof(double) * BD, cudaMemcpyDefault));
    for (size_t b = 0; b < B; ++b)
        if (int r = build_ties((int)b, (int)D, c->N, ms.data() + b * D, sc.data() + b * D, of.data() + b * D,
                               h.data() + b * D, box.data() + b * D, box.data() + BD + b * D,
                               ti.data() + b * (3 * D + 2), td.data() + b * 2 * D, h.data() + 2 * BD + b * D,
                               h.data() + 3 * BD + b * D))
            return r;
    std::copy(h.begin(), h.begin() + BD, h.begin() + BD);
    CK(c->rf_tie_i.reserve(ti.size()));
    CK(c->rf_tie_d.reserve(td.size()));
    CK(cudaMemcpyAsync(c->rf_tie_i.ptr, ti.data(), sizeof(int) * ti.size(), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->rf_tie_d.ptr, td.data(), sizeof(double) * td.size(), cudaMemcpyHostToDevice, st));
    const RefineTies ties{c->rf_tie_i.ptr, c->rf_tie_d.ptr};
    return refine_run(c, h, &ties, loss, fscale, max_iter, xtol, x, f_out, passes_out, accepted_out, status_out, st);
}

int nmrfit_ctx_refine_loss(nmrfit_ctx* c, double* x, const double* lb, const double* ub, const int* tie_master,
                           const double* tie_scale, const double* tie_offset, int loss, const double* f_scale,
                           int max_iter, double xtol, double* f_out, int* passes_out, int* accepted_out,
                           int* status_out, void* stream) {
    const int n_tie = (tie_master != nullptr) + (tie_scale != nullptr) + (tie_offset != nullptr);
    const bool tied = n_tie == 3;
    cudaStream_t st = (cudaStream_t)stream;
    const double* unused = nullptr;
    if (int r = post_fit_begin(
            c,
            [&] {
                if (!x || !lb || !ub) return fail(NMRFIT_ERR_ARG, "x, lb and ub must be non-NULL");
                if (n_tie != 0 && n_tie != 3)
                    return fail(NMRFIT_ERR_ARG, "tie_master, tie_scale and tie_offset must be all NULL (untied) or "
                                                "all non-NULL");
                return check_loss(loss);
            },
            "refinement supports", [&] { return refine_check(c, max_iter, xtol, tied); }, "it is refined", nullptr, st,
            &unused))
        return r;
    const double* fs = nullptr;
    if (int r = stage_loss(c, loss, f_scale, st, &fs)) return r;
    if (tied)
        return refine_tied(c, x, lb, ub, tie_master, tie_scale, tie_offset, loss, fs, max_iter, xtol, f_out,
                           passes_out, accepted_out, status_out, st);
    return refine_untied(c, x, lb, ub, loss, fs, max_iter, xtol, f_out, passes_out, accepted_out, status_out, st);
}

// the least-squares refinements: nmrfit_ctx_refine_loss with LINEAR, past their own NULL checks
int nmrfit_ctx_refine(nmrfit_ctx* c, double* x, const double* lb, const double* ub, int max_iter, double xtol,
                      double* f_out, int* passes_out, int* accepted_out, int* status_out, void* stream) {
    if (int r = check_ctx(c)) return r;
    if (!x || !lb || !ub) return fail(NMRFIT_ERR_ARG, "x, lb and ub must be non-NULL");
    return nmrfit_ctx_refine_loss(c, x, lb, ub, nullptr, nullptr, nullptr, NMRFIT_LOSS_LINEAR, nullptr, max_iter, xtol,
                                  f_out, passes_out, accepted_out, status_out, stream);
}

int nmrfit_ctx_refine_tied(nmrfit_ctx* c, double* x, const double* lb, const double* ub, const int* tie_master,
                           const double* tie_scale, const double* tie_offset, int max_iter, double xtol, double* f_out,
                           int* passes_out, int* accepted_out, int* status_out, void* stream) {
    if (int r = check_ctx(c)) return r;
    if (!x || !lb || !ub || !tie_master || !tie_scale || !tie_offset)
        return fail(NMRFIT_ERR_ARG, "x, lb, ub, tie_master, tie_scale and tie_offset must be non-NULL");
    return nmrfit_ctx_refine_loss(c, x, lb, ub, tie_master, tie_scale, tie_offset, NMRFIT_LOSS_LINEAR, nullptr,
                                  max_iter, xtol, f_out, passes_out, accepted_out, status_out, stream);
}

int nmrfit_normal_eq_plan(int n_points, int n_peaks, int* out) {
    if (!out) return fail(NMRFIT_ERR_ARG, "out is NULL");
    if (n_peaks < 1 || n_peaks > 64) return fail(NMRFIT_ERR_ARG, "n_peaks must be 1..64");
    if (n_points < 1) return fail(NMRFIT_ERR_ARG, "n_points must be >= 1");
    const NormalEqPlan p = normal_eq_plan(n_points, n_peaks);
    const int v[10] = {p.ng, p.slices, p.tasks, p.tasks_per_slice, p.threads, p.tp, p.chunk, p.n_chunks,
                       (int)p.smem, (int)normal_eq_scratch_doubles(p, 1)};
    for (int k = 0; k < 10; ++k) out[k] = v[k];
    return NMRFIT_OK;
}

int nmrfit_ctx_set_algorithm(nmrfit_ctx* c, int algorithm) {
    if (int r = check_ctx(c)) return r;
    if (algorithm != NMRFIT_ALGO_AUTO && algorithm != NMRFIT_ALGO_GENERAL && algorithm != NMRFIT_ALGO_UNIFORM)
        return fail(NMRFIT_ERR_ARG, "algorithm must be NMRFIT_ALGO_AUTO, _GENERAL or _UNIFORM");
    c->algorithm = algorithm;
    return NMRFIT_OK;
}

int nmrfit_ctx_get_algorithm(nmrfit_ctx* c, int fit_im, int* algorithm) {
    if (int r = check_ctx(c)) return r;
    if (!algorithm) return fail(NMRFIT_ERR_ARG, "algorithm is NULL");
    const int k = ctx_plan(c, 1, fit_im).kernel;
    *algorithm = k == OBJ_GENERAL || k == OBJ_F32_GENERAL ? NMRFIT_ALGO_GENERAL : NMRFIT_ALGO_UNIFORM;
    return NMRFIT_OK;
}

int nmrfit_ctx_set_tuning(nmrfit_ctx* c, int threads, int r, int tb, int sp) {
    if (int rc = check_ctx(c)) return rc;
    if (threads != 0 && threads != 128 && threads != 256) return fail(NMRFIT_ERR_ARG, "threads must be 0, 128 or 256");
    if (r != 0 && r != 2 && r != 4 && r != 8 && r != 16)
        return fail(NMRFIT_ERR_ARG, "points_per_thread must be 0, 2, 4, 8 or 16");
    if (tb != 0 && tb != 6 && tb != 8 && tb != 10 && tb != -1)
        return fail(NMRFIT_ERR_ARG, "exp_table_bits must be 0 (auto), -1 (no table), 6, 8 or 10");
    if (sp < 0 || sp > 64) return fail(NMRFIT_ERR_ARG, "particles_per_cta must be 0..64");
    c->user_tune.threads = threads; c->user_tune.r = r; c->user_tune.tb = tb; c->user_tune.sp = sp;
    return NMRFIT_OK;
}

int nmrfit_ctx_set_variant(nmrfit_ctx* c, int variant, int stages, int occupancy) {
    if (int rc = check_ctx(c)) return rc;
    if (variant < -1 || variant > 1) return fail(NMRFIT_ERR_ARG, "variant must be -1 (auto), 0 (one group per CTA) or 1 (streamed)");
    if (stages != 0 && (stages < 2 || stages > 4)) return fail(NMRFIT_ERR_ARG, "stages must be 0 (auto) or 2..4");
    if (occupancy != 0 && occupancy != 2 && occupancy != 3) return fail(NMRFIT_ERR_ARG, "occupancy must be 0 (auto), 2 or 3");
    c->user_tune.variant = variant;
    c->user_tune.stages = stages;
    c->user_tune.occ = occupancy;
    return NMRFIT_OK;
}

int nmrfit_ctx_set_far_cells(nmrfit_ctx* c, int cells) {
    if (int rc = check_ctx(c)) return rc;
    if (cells != 0 && cells != 1 && cells != 2 && cells != 4) return fail(NMRFIT_ERR_ARG, "cells must be 0 (auto), 1, 2 or 4");
    c->far_cells = cells;
    return NMRFIT_OK;
}

int nmrfit_ctx_get_variant(nmrfit_ctx* c, int S, int* variant, int* stages) {
    if (int rc = check_ctx(c)) return rc;
    const ObjTune t = ctx_plan(c, S < 1 ? 1 : S, NMRFIT_REAL_ONLY).t;
    if (variant) *variant = t.variant;
    if (stages) *stages = t.stages;
    return NMRFIT_OK;
}

int nmrfit_ctx_get_tuning(nmrfit_ctx* c, int S, int* threads, int* r, int* tb, int* sp, int* n_tiles) {
    if (int rc = check_ctx(c)) return rc;
    const ObjPlan p = ctx_plan(c, S < 1 ? 1 : S, NMRFIT_REAL_ONLY);
    const ObjTune& t = p.t;
    if (threads) *threads = t.threads;
    if (r) *r = t.r;
    if (tb) *tb = t.tb;
    if (sp) *sp = t.sp;
    if (n_tiles) *n_tiles = p.n_tiles;
    return NMRFIT_OK;
}

int nmrfit_ctx_set_fused(nmrfit_ctx* c, int mode) {
    if (int rc = check_ctx(c)) return rc;
    if (mode != NMRFIT_FUSED_AUTO && mode != NMRFIT_FUSED_OFF && mode != NMRFIT_FUSED_REQUIRE)
        return fail(NMRFIT_ERR_ARG, "mode must be NMRFIT_FUSED_AUTO, _OFF or _REQUIRE");
    c->fused_mode = mode;
    return NMRFIT_OK;
}

int nmrfit_ctx_fused_timing(nmrfit_ctx* c, int enable, long long* cycles) {
    if (int rc = check_ctx(c)) return rc;
    CK(cudaSetDevice(c->device));
    if (cycles) {
        if (!c->ftiming.ptr) return fail(NMRFIT_ERR_STATE, "fused timing was not enabled");
        CK(cudaDeviceSynchronize());
        CK(cudaMemcpy(cycles, c->ftiming.ptr, sizeof(long long) * 8, cudaMemcpyDeviceToHost));
    }
    c->fused_timing = enable != 0;
    if (c->fused_timing) {
        CK(c->ftiming.reserve(8));
        CK(cudaMemset(c->ftiming.ptr, 0, sizeof(long long) * 8));
    }
    return NMRFIT_OK;
}

int nmrfit_ctx_fused_launches(nmrfit_ctx* c, long long* launches) {
    if (int rc = check_ctx(c)) return rc;
    if (!launches) return fail(NMRFIT_ERR_ARG, "launches is NULL");
    *launches = c->fused_launches;
    return NMRFIT_OK;
}

int nmrfit_ctx_profile(nmrfit_ctx* c, int enable) {
    if (int rc = check_ctx(c)) return rc;
    c->profiling = enable != 0;
    c->prof_used = 0;
    return NMRFIT_OK;
}

int nmrfit_ctx_profile_read_split(nmrfit_ctx* c, double* prepare_ms, double* evaluate_ms, long long* launches) {
    if (int rc = check_ctx(c)) return rc;
    CK(cudaSetDevice(c->device));
    double prep = 0.0, eval = 0.0;
    for (size_t i = 0; i + 2 < c->prof_used; i += 3) {
        CK(cudaEventSynchronize(c->prof_events[i + 2].h));
        float a = 0.f, b = 0.f;
        CK(cudaEventElapsedTime(&a, c->prof_events[i].h, c->prof_events[i + 1].h));
        CK(cudaEventElapsedTime(&b, c->prof_events[i + 1].h, c->prof_events[i + 2].h));
        prep += a;
        eval += b;
    }
    if (prepare_ms) *prepare_ms = prep;
    if (evaluate_ms) *evaluate_ms = eval;
    if (launches) *launches = (long long)(c->prof_used / 3);
    c->prof_used = 0;
    return NMRFIT_OK;
}

int nmrfit_ctx_profile_read(nmrfit_ctx* c, double* total_ms, long long* launches) {
    double prep = 0.0, eval = 0.0;
    if (int rc = nmrfit_ctx_profile_read_split(c, &prep, &eval, launches)) return rc;
    if (total_ms) *total_ms = prep + eval;
    return NMRFIT_OK;
}

int nmrfit_objective_batch(nmrfit_ctx* c, const double* x_dev, int S, int fit_im, double* f_dev, void* stream) {
    if (int rc = check_ctx(c)) return rc;
    if (!x_dev || !f_dev) return fail(NMRFIT_ERR_ARG, "x_dev and f_dev must be non-NULL");
    if (S < 1) return fail(NMRFIT_ERR_ARG, "n_particles must be >= 1");
    CK(cudaSetDevice(c->device));
    return run_objective(c, x_dev, S, fit_im, f_dev, (cudaStream_t)stream);
}

namespace {
// Page-locked host positions as the device sees them (null: pageable memory, or a path without the prepare pass)
const double* mapped_positions(const nmrfit_ctx* c, const double* x_host, int S, int fit_im) {
    if (!two_pass(ctx_plan(c, S, fit_im))) return nullptr;
    cudaPointerAttributes at{};
    const cudaError_t pe = cudaPointerGetAttributes(&at, x_host);
    if (pe != cudaSuccess) (void)cudaGetLastError();
    return (pe == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) ? (const double*)at.devicePointer : nullptr;
}
}  // namespace

int nmrfit_objective_batch_host(nmrfit_ctx* c, const double* x_host, int S, int fit_im, double* f_host) {
    if (int rc = check_ctx(c)) return rc;
    if (!x_host || !f_host) return fail(NMRFIT_ERR_ARG, "x_host and f_host must be non-NULL");
    if (S < 1) return fail(NMRFIT_ERR_ARG, "n_particles must be >= 1");
    CK(cudaSetDevice(c->device));
    size_t nx = (size_t)c->B * S * c->D, nf = (size_t)c->B * S;
    CK(c->x_stage.reserve(nx));
    CK(c->f_stage.reserve(nf));
    // A large particle set of one spectrum goes through in slices on two streams: while slice k is evaluated, slice
    // k + 1's positions are on their way in and slice k - 1's values on their way out (each slice has its own scratch).
    // Page-locked host positions (cudaHostAlloc / cudaHostRegister: mapped into the device under unified addressing) are
    // read by the prepare pass ITSELF, each element crossing PCIe once while other CTAs compute - no staging copy in
    // front of the kernels.  Pageable arrays take the copies below.
    const double* x_map = mapped_positions(c, x_host, S, fit_im);     // the caller's array as the device sees it, or null
    constexpr int kPad = 64;
    // (slices of ~12k particles, two to six of them: 1.24 / 1.15 / 1.13 / 1.12 ms per call with 1 / 2 / 4 / 6 slices
    // at 65,536 particles of 6 peaks x 4,096 points, tools/e2e_probe.py)
    // (in-place reads are not sliced: 1.048 / 1.084 / 1.105 ms with 1 / 2 / 3 slices - and 1.136 ms for the best copy path)
    const int kSlices = x_map ? 1 : std::min(6, std::max(2, S / 12288));
    if (c->B == 1 && S >= 4 * 4096 && !c->profiling && kSlices > 1) {
        for (Stream& ps : c->pipe) CK(ensure_stream(ps));
        CK(c->h_f.reserve(nf));
        const int chunk = ((S + kSlices - 1) / kSlices + 63) & ~63;
        const size_t total = (size_t)kSlices * (chunk + kPad);
        for (int k = 0, s0 = 0; s0 < S; ++k, s0 += chunk) {
            const int ns = std::min(chunk, S - s0);
            cudaStream_t ps = c->pipe[k & 1].h;
            if (!x_map)
                CK(cudaMemcpyAsync(c->x_stage.ptr + (size_t)s0 * c->D, x_host + (size_t)s0 * c->D, sizeof(double) * ns * c->D,
                                   cudaMemcpyHostToDevice, ps));
            const ObjIn slice{x_map ? x_map + (size_t)s0 * c->D : nullptr, (size_t)k * (chunk + kPad), total};
            if (int rc = run_objective(c, c->x_stage.ptr + (size_t)s0 * c->D, ns, fit_im, c->f_stage.ptr + s0, ps, slice))
                return rc;
            // (into page-locked staging: an "async" copy into the caller's pageable array would block the host until
            // the slice has been evaluated, and the slices would run one after the other)
            CK(cudaMemcpyAsync(c->h_f.ptr + s0, c->f_stage.ptr + s0, sizeof(double) * ns, cudaMemcpyDeviceToHost, ps));
        }
        for (Stream& ps : c->pipe) CK(cudaStreamSynchronize(ps.h));
        std::memcpy(f_host, c->h_f.ptr, sizeof(double) * nf);
        return NMRFIT_OK;
    }
    cudaStream_t st = 0;
    if (!x_map) CK(cudaMemcpyAsync(c->x_stage.ptr, x_host, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    if (int rc = run_objective(c, c->x_stage.ptr, S, fit_im, c->f_stage.ptr, st, ObjIn{x_map})) return rc;
    CK(cudaMemcpyAsync(f_host, c->f_stage.ptr, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return NMRFIT_OK;
}

// equations.objective's own calling convention - the spectrum comes along with every call - for one spectrum:
// nmrfit_ctx_set_spectrum + nmrfit_objective_batch_host in one.  When the context already holds a spectrum and the
// positions are page-locked, the kernels are launched FIRST, on the spectrum the device has, and the four arrays are
// compared with the host copy while they run (1 MB at 32,768 points: ~60 us that used to sit in front of every call);
// a spectrum that did change is uploaded and the evaluation repeated.
int nmrfit_objective_spectrum_host(nmrfit_ctx* c, const double* w, const double* u, const double* v, const double* weights,
                                   const double* x_host, int S, int fit_im, double* f_host) {
    if (int rc = check_ctx(c)) return rc;
    if (c->B != 1) return fail(NMRFIT_ERR_ARG, "nmrfit_objective_spectrum_host is for contexts of one spectrum");
    if (!w || !u || !v || !weights || !x_host || !f_host) return fail(NMRFIT_ERR_ARG, "NULL argument");
    if (S < 1) return fail(NMRFIT_ERR_ARG, "n_particles must be >= 1");
    CK(cudaSetDevice(c->device));
    const size_t N = (size_t)c->N;
    const bool have = c->spec_set[0] && !c->shadow.empty() && c->shadow[0].size() == 4 * N && !is_device_pointer(w) &&
                      !is_device_pointer(u) && !is_device_pointer(v) && !is_device_pointer(weights);
    const double* x_map = have && !c->profiling ? mapped_positions(c, x_host, S, fit_im) : nullptr;
    if (!x_map) {
        if (int rc = nmrfit_ctx_set_spectrum(c, 0, w, u, v, weights)) return rc;
        return nmrfit_objective_batch_host(c, x_host, S, fit_im, f_host);
    }
    CK(c->x_stage.reserve((size_t)S * c->D));
    CK(c->f_stage.reserve((size_t)S));
    cudaStream_t st = 0;
    if (int rc = run_objective(c, c->x_stage.ptr, S, fit_im, c->f_stage.ptr, st, ObjIn{x_map})) return rc;
    const double* src[4] = {w, u, v, weights};
    bool same = true;
    for (int k = 0; same && k < 4; ++k) same = std::memcmp(c->shadow[0].data() + (size_t)k * N, src[k], sizeof(double) * N) == 0;
    if (!same) {
        CK(cudaStreamSynchronize(st));                     // the speculative evaluation is dropped
        if (int rc = nmrfit_ctx_set_spectrum(c, 0, w, u, v, weights)) return rc;
        return nmrfit_objective_batch_host(c, x_host, S, fit_im, f_host);
    }
    CK(cudaMemcpyAsync(f_host, c->f_stage.ptr, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return NMRFIT_OK;
}

// ---- swarm ---------------------------------------------------------------------------------------

int nmrfit_pso_begin(nmrfit_ctx* c, const double* lb, const double* ub, const nmrfit_pso_opts* o, const double* r_pos,
                     const double* r_vel, void* stream) {
    if (int rc = check_ctx(c)) return rc;
    if (!lb || !ub || !o) return fail(NMRFIT_ERR_ARG, "lb, ub and opts must be non-NULL");
    if (o->swarmsize < 1) return fail(NMRFIT_ERR_ARG, "swarmsize must be >= 1");
    if (o->maxiter < 0) return fail(NMRFIT_ERR_ARG, "maxiter must be >= 0");
    if (o->fit_im < 0 || o->fit_im > 2) return fail(NMRFIT_ERR_ARG, "fit_im must be 0, 1 or 2");
    const int B = c->B, S = o->swarmsize, D = c->D;
    const int nb = o->bounds_per_spectrum ? B : 1;
    for (int i = 0; i < nb * D; ++i)      // pyswarm: assert np.all(ub > lb)
        if (!(ub[i] > lb[i])) return fail(NMRFIT_ERR_ARG, "All upper-bound values must be greater than lower-bound values");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    size_t nsd = (size_t)B * S * D, ns = (size_t)B * S;
    CK(c->sx.reserve(nsd)); CK(c->sv.reserve(nsd)); CK(c->sp.reserve(nsd));
    CK(c->sfx.reserve(ns)); CK(c->sfp.reserve(ns));
    CK(c->sg.reserve((size_t)B * D)); CK(c->sfg.reserve(B)); CK(c->sbx.reserve((size_t)B * D)); CK(c->sbf.reserve(B));
    CK(c->slb.reserve((size_t)B * D)); CK(c->sub.reserve((size_t)B * D)); CK(c->srec.reserve((size_t)B * (D + 2)));
    CK(c->sstop.reserve(B)); CK(c->sit.reserve(B));
    CK(c->fin_scratch.reserve(swarm_finish_scratch_doubles(B, S)));
    CK(c->fin_tickets.reserve(B));
    CK(cudaMemsetAsync(c->fin_tickets.ptr, 0, sizeof(unsigned) * B, (cudaStream_t)stream));
    std::vector<double> hl((size_t)B * D), hu((size_t)B * D);
    for (int b = 0; b < B; ++b)
        for (int d = 0; d < D; ++d) {
            hl[(size_t)b * D + d] = lb[(o->bounds_per_spectrum ? (size_t)b * D : 0) + d];
            hu[(size_t)b * D + d] = ub[(o->bounds_per_spectrum ? (size_t)b * D : 0) + d];
        }
    CK(cudaMemcpyAsync(c->slb.ptr, hl.data(), hl.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(c->sub.ptr, hu.data(), hu.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));      // hl/hu go out of scope
    CK(cudaMemsetAsync(c->sstop.ptr, 0, sizeof(int) * B, st));
    CK(cudaMemsetAsync(c->sit.ptr, 0, sizeof(int) * B, st));
    SwarmState& s = c->sw;
    s.B = B; s.S = S; s.D = D;
    s.x = c->sx.ptr; s.v = c->sv.ptr; s.p = c->sp.ptr; s.fx = c->sfx.ptr; s.fp = c->sfp.ptr;
    s.g = c->sg.ptr; s.fg = c->sfg.ptr; s.best_x = c->sbx.ptr; s.best_f = c->sbf.ptr;
    s.lb = c->slb.ptr; s.ub = c->sub.ptr; s.rec = c->srec.ptr; s.stop = c->sstop.ptr; s.it = c->sit.ptr;
    s.omega = o->omega; s.phip = o->phip; s.phig = o->phig; s.minstep = o->minstep; s.minfunc = o->minfunc;
    s.seed = o->seed; s.index0 = o->particle_offset; s.spec0 = o->spectrum_offset;
    c->maxiter = o->maxiter; c->kk = o->fit_im; c->generation = 0; c->swarm = true;
    c->epoch += 1;

    const double *rp_d = nullptr, *rv_d = nullptr;
    if (int rc = stage(r_pos, nsd, c->rnd_a, st, &rp_d)) return rc;
    if (int rc = stage(r_vel, nsd, c->rnd_b, st, &rv_d)) return rc;
    cudaError_t e = launch_swarm_init(s, rp_d, nullptr, st);
    if (e == cudaSuccess) e = launch_swarm_init_velocity(s, rv_d, st);
    if (e != cudaSuccess) return fail_cuda(e, "swarm init");
    return swarm_generation(c, false, nullptr, nullptr, 0, st);
}

namespace {
// One generation of nmrfit_pso_advance (commit 0), nmrfit_pso_step (1) or nmrfit_pso_step_peers (2)
int pso_generation(nmrfit_ctx* c, const double* rp, const double* rg, int commit, void* stream) {
    if (int rc = require_swarm(c)) return rc;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const double *rp_d, *rg_d;
    if (int rc = stage_random(c, 1, rp, rg, "rp and rg", st, &rp_d, &rg_d)) return rc;
    return queue_generations(c, 1, rp_d, rg_d, commit, st);
}

// the argument checks of nmrfit_ctx_mt19937 and nmrfit_ctx_mt19937_begin
int mt_check(const nmrfit_ctx* c, int pos, long long n_arrays) {
    if (pos < 0 || pos > 624) return fail(NMRFIT_ERR_ARG, "MT19937 position must be 0..624");
    if (n_arrays < 2 || (n_arrays & 1)) return fail(NMRFIT_ERR_ARG, "n_arrays must be even: arrays come in (first, second) pairs");
    if (c->mt_elems == 0) return fail(NMRFIT_ERR_STATE, "call nmrfit_ctx_mt19937_shape first");
    return NMRFIT_OK;
}

// Queue on `st` the generation of n_arrays arrays into (a, b) in turn, from the state (key [624] + position) at
// `state_in`; the advanced state goes back to `state_out`.  Each caller has its own buffers: nmrfit_ctx_mt19937 may
// run while a nmrfit_ctx_mt19937_begin is pending.
int mt_queue(nmrfit_ctx* c, long long n_arrays, DevBuf<double>& a, DevBuf<double>& b, DevBuf<unsigned>& state,
             DevBuf<unsigned>& words, const unsigned* state_in, unsigned* state_out, cudaStream_t st) {
    const long long nsd = c->mt_elems, pairs = n_arrays / 2;
    CK(a.reserve((size_t)(pairs * nsd)));
    CK(b.reserve((size_t)(pairs * nsd)));
    CK(state.reserve(625));
    CK(words.reserve((size_t)(2 * n_arrays * nsd)));
    CK(cudaMemcpyAsync(state.ptr, state_in, sizeof(unsigned) * 625, cudaMemcpyHostToDevice, st));
    cudaError_t e = launch_mt19937(state.ptr, reinterpret_cast<int*>(state.ptr + 624), n_arrays * nsd, words.ptr, a.ptr,
                                   b.ptr, nsd, st);
    if (e != cudaSuccess) return fail_cuda(e, "MT19937 launch");
    CK(cudaMemcpyAsync(state_out, state.ptr, sizeof(unsigned) * 625, cudaMemcpyDeviceToHost, st));
    return NMRFIT_OK;
}
}  // namespace

int nmrfit_pso_advance(nmrfit_ctx* c, const double* rp, const double* rg, void* stream) {
    return pso_generation(c, rp, rg, 0, stream);
}

int nmrfit_pso_step(nmrfit_ctx* c, const double* rp, const double* rg, void* stream) {
    return pso_generation(c, rp, rg, 1, stream);
}

int nmrfit_ctx_mt19937(nmrfit_ctx* c, unsigned* key, int* pos, long long n_arrays, double** a_dev, double** b_dev,
                       void* stream) {
    if (int rc = check_ctx(c)) return rc;
    if (!key || !pos || !a_dev || !b_dev) return fail(NMRFIT_ERR_ARG, "NULL argument");
    if (int rc = mt_check(c, *pos, n_arrays)) return rc;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned host[625];
    std::memcpy(host, key, sizeof(unsigned) * 624);
    host[624] = (unsigned)*pos;
    if (int rc = mt_queue(c, n_arrays, c->rnd_a, c->rnd_b, c->mt_state, c->mt_words, host, host, st)) return rc;
    CK(cudaStreamSynchronize(st));
    std::memcpy(key, host, sizeof(unsigned) * 624);
    *pos = (int)host[624];
    *a_dev = c->rnd_a.ptr;
    *b_dev = c->rnd_b.ptr;
    return NMRFIT_OK;
}

// The same in two halves, on a stream of the context's own: `begin` queues the generation and returns at once, `end`
// waits for it and hands back the advanced state.  Between the two the caller runs the swarm on the PREVIOUS set of
// arrays - the sequential recurrence (one CTA, ~0.2 us per 227 words) hides behind the fit's kernels.  Two sets of
// arrays are used in turn: the pointers of one `begin` stay valid until the `begin` after the next.
int nmrfit_ctx_mt19937_begin(nmrfit_ctx* c, const unsigned* key, int pos, long long n_arrays, double** a_dev, double** b_dev) {
    if (int rc = check_ctx(c)) return rc;
    if (!key || !a_dev || !b_dev) return fail(NMRFIT_ERR_ARG, "NULL argument");
    if (int rc = mt_check(c, pos, n_arrays)) return rc;
    if (c->mt_pending) return fail(NMRFIT_ERR_STATE, "nmrfit_ctx_mt19937_end has not been called for the previous begin");
    CK(cudaSetDevice(c->device));
    CK(ensure_stream(c->mt_stream));
    CK(c->mt_host.reserve(2 * 625));
    const int k = c->mt_flip;
    std::memcpy(c->mt_host.ptr, key, sizeof(unsigned) * 624);
    c->mt_host.ptr[624] = (unsigned)pos;
    // (growing a buffer frees and allocates: an implicit device synchronisation, first calls only)
    if (int rc = mt_queue(c, n_arrays, c->mt_a[k], c->mt_b[k], c->mt_state2, c->mt_words2, c->mt_host.ptr,
                          c->mt_host.ptr + 625, c->mt_stream.h))
        return rc;
    *a_dev = c->mt_a[k].ptr;
    *b_dev = c->mt_b[k].ptr;
    c->mt_flip ^= 1;
    c->mt_pending = 1;
    return NMRFIT_OK;
}

int nmrfit_ctx_mt19937_end(nmrfit_ctx* c, unsigned* key_out, int* pos_out) {
    if (int rc = check_ctx(c)) return rc;
    if (!c->mt_pending) return fail(NMRFIT_ERR_STATE, "no nmrfit_ctx_mt19937_begin is pending");
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->mt_stream.h));
    c->mt_pending = 0;
    if (key_out) std::memcpy(key_out, c->mt_host.ptr + 625, sizeof(unsigned) * 624);
    if (pos_out) *pos_out = (int)c->mt_host.ptr[625 + 624];
    return NMRFIT_OK;
}

int nmrfit_ctx_mt19937_shape(nmrfit_ctx* c, long long elements_per_array) {
    if (int rc = check_ctx(c)) return rc;
    if (elements_per_array < 1) return fail(NMRFIT_ERR_ARG, "elements_per_array must be >= 1");
    c->mt_elems = elements_per_array;
    return NMRFIT_OK;
}

// ---- record exchange over peer memory -------------------------------------------------------------

int nmrfit_pso_peer_export(nmrfit_ctx* c, int n_ranks, int rank, void* ipc_handle_out, void** base_out) {
    if (int rc = check_ctx(c)) return rc;
    if (n_ranks < 1 || n_ranks > 64 || rank < 0 || rank >= n_ranks) return fail(NMRFIT_ERR_ARG, "bad rank / n_ranks");
    if (c->peer_win.h) return fail(NMRFIT_ERR_STATE, "the exchange window of this context already exists");
    CK(cudaSetDevice(c->device));
    const size_t W = (size_t)c->D + 2;
    c->peer_rec_bytes = (2 * (size_t)n_ranks * c->B * W * sizeof(double) + 15) & ~(size_t)15;
    // CUDA IPC exports the whole backing block of an allocation: the window gets blocks of its own (a multiple of the
    // 2 MiB granule), so that a peer that opens the handle cannot reach any other allocation of this process
    const size_t granule = (size_t)2 << 20;
    const size_t bytes = ((c->peer_rec_bytes + (size_t)n_ranks * c->B * sizeof(long long) + granule - 1) / granule) * granule;
    CK(cudaMalloc(&c->peer_win.h, bytes));
    CK(cudaMemset(c->peer_win.h, 0, bytes));               // tokens start at 0; the first real token is (1 << 32)
    CK(cudaDeviceSynchronize());
    c->peer_ranks = n_ranks;
    c->peer_rank = rank;
    if (ipc_handle_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, c->peer_win.h));
        std::memcpy(ipc_handle_out, &h, sizeof(h));
    }
    if (base_out) *base_out = c->peer_win.h;
    return NMRFIT_OK;
}

int nmrfit_pso_peer_open(nmrfit_ctx* c, const void* ipc_handles, void* const* local_bases) {
    if (int rc = check_ctx(c)) return rc;
    if (!c->peer_win.h) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_peer_export has not been called");
    if (!ipc_handles && !local_bases) return fail(NMRFIT_ERR_ARG, "ipc_handles or local_bases must be given");
    CK(cudaSetDevice(c->device));
    const int R = c->peer_ranks;
    std::vector<double*> recs(R);
    std::vector<long long*> toks(R);
    for (int q = 0; q < R; ++q) {
        void* base = nullptr;
        if (q == c->peer_rank) {
            base = c->peer_win.h;
        } else if (local_bases && local_bases[q]) {
            base = local_bases[q];                          // another context of this process
        } else {
            cudaIpcMemHandle_t h;
            std::memcpy(&h, (const char*)ipc_handles + (size_t)q * sizeof(h), sizeof(h));
            CK(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
            c->peer_opened.emplace_back(base);
        }
        recs[q] = (double*)base;
        toks[q] = (long long*)((char*)base + c->peer_rec_bytes);
    }
    CK(c->peer_recs_dev.reserve(R));
    CK(c->peer_tok_dev.reserve(R));
    CK(c->peer_err.reserve(1));
    CK(cudaMemcpy(c->peer_recs_dev.ptr, recs.data(), sizeof(double*) * R, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->peer_tok_dev.ptr, toks.data(), sizeof(long long*) * R, cudaMemcpyHostToDevice));
    CK(cudaMemset(c->peer_err.ptr, 0, sizeof(int)));
    c->peers_ready = true;
    return NMRFIT_OK;
}

namespace {
int exchange_commit(nmrfit_ctx* c, cudaStream_t st) {
    if (!c->peers_ready) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_peer_open has not been called");
    const PeerArgs pa = make_peer_args(c);
    cudaError_t e = launch_swarm_exchange_commit(c->sw, pa, c->generation == 0, c->maxiter, st);
    if (e != cudaSuccess) return fail_cuda(e, "exchange + commit launch");
    return NMRFIT_OK;
}
}  // namespace

int nmrfit_pso_commit_peers(nmrfit_ctx* c, void* stream) {
    if (int rc = require_swarm(c)) return rc;
    CK(cudaSetDevice(c->device));
    return exchange_commit(c, (cudaStream_t)stream);
}

int nmrfit_pso_step_peers(nmrfit_ctx* c, const double* rp, const double* rg, void* stream) {
    return pso_generation(c, rp, rg, 2, stream);
}

int nmrfit_pso_run_peers(nmrfit_ctx* c, int n_generations, const double* rp_all, const double* rg_all, int* n_running,
                         int* timed_out, void* stream) {
    if (int rc = require_swarm(c)) return rc;
    if (n_generations < 0) return fail(NMRFIT_ERR_ARG, "n_generations must be >= 0");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const double *rp_d, *rg_d;
    if (int rc = stage_random(c, n_generations, rp_all, rg_all, "rp_all and rg_all", st, &rp_d, &rg_d)) return rc;
    if (int rc = queue_generations(c, n_generations, rp_d, rg_d, 2, st)) return rc;
    if (int rc = queue_stop_flags(c, c->peer_err.ptr, st)) return rc;
    CK(cudaStreamSynchronize(st));
    if (n_running) *n_running = running_spectra(c);
    if (timed_out) *timed_out = c->h_flags.ptr[c->sw.B];
    return NMRFIT_OK;
}

// ---- the same for the contexts of ONE process (a C consumer with one context per GPU and no NCCL) -------------------

int nmrfit_comm_init_all(nmrfit_ctx* const* ctxs, int n) {
    if (!ctxs || n < 1 || n > 64) return fail(NMRFIT_ERR_ARG, "ctxs must hold 1..64 contexts");
    for (int r = 0; r < n; ++r) {
        if (int rc = check_ctx(ctxs[r])) return rc;
        if (ctxs[r]->B != ctxs[0]->B || ctxs[r]->D != ctxs[0]->D)
            return fail(NMRFIT_ERR_ARG, "the contexts of a communicator must agree in spectra and parameters");
    }
    // every device stores into every other device's window
    for (int r = 0; r < n; ++r) {
        CK(cudaSetDevice(ctxs[r]->device));
        for (int q = 0; q < n; ++q) {
            if (ctxs[q]->device == ctxs[r]->device) continue;
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, ctxs[r]->device, ctxs[q]->device));
            if (!can) return fail(NMRFIT_ERR_STATE, "the devices of the communicator cannot reach each other's memory");
            const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) (void)cudaGetLastError();
            else if (e != cudaSuccess) return fail_cuda(e, "cudaDeviceEnablePeerAccess");
        }
    }
    std::vector<void*> bases(n, nullptr);
    for (int r = 0; r < n; ++r)
        if (int rc = nmrfit_pso_peer_export(ctxs[r], n, r, nullptr, &bases[r])) return rc;
    for (int r = 0; r < n; ++r)
        if (int rc = nmrfit_pso_peer_open(ctxs[r], nullptr, bases.data())) return rc;
    return NMRFIT_OK;
}

namespace {
int comm_stream(nmrfit_ctx* c, cudaStream_t* st) {
    CK(cudaSetDevice(c->device));
    CK(ensure_stream(c->pipe[0]));
    CK(cudaStreamSynchronize(0));                          // nmrfit_pso_begin and friends ran on the default stream
    *st = c->pipe[0].h;
    return NMRFIT_OK;
}
}  // namespace

int nmrfit_comm_commit(nmrfit_ctx* const* ctxs, int n) {
    if (!ctxs || n < 1) return fail(NMRFIT_ERR_ARG, "ctxs must hold at least one context");
    for (int r = 0; r < n; ++r) {
        if (int rc = check_ctx(ctxs[r])) return rc;
        if (!ctxs[r]->swarm) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_begin has not been called on every context");
    }
    for (int r = 0; r < n; ++r) {                           // all launched before any is waited for: they wait for each other
        cudaStream_t st;
        if (int rc = comm_stream(ctxs[r], &st)) return rc;
        if (int rc = exchange_commit(ctxs[r], st)) return rc;
    }
    for (int r = 0; r < n; ++r) {
        CK(cudaSetDevice(ctxs[r]->device));
        CK(cudaStreamSynchronize(ctxs[r]->pipe[0].h));
    }
    return NMRFIT_OK;
}

int nmrfit_comm_run(nmrfit_ctx* const* ctxs, int n, int n_generations, const double* const* rp_all,
                    const double* const* rg_all, int* n_running, int* timed_out) {
    if (!ctxs || n < 1) return fail(NMRFIT_ERR_ARG, "ctxs must hold at least one context");
    if (n_generations < 0) return fail(NMRFIT_ERR_ARG, "n_generations must be >= 0");
    std::vector<const double*> rp_d(n), rg_d(n);
    std::vector<cudaStream_t> sts(n);
    for (int r = 0; r < n; ++r) {
        nmrfit_ctx* c = ctxs[r];
        if (int rc = check_ctx(c)) return rc;
        if (!c->swarm) return fail(NMRFIT_ERR_STATE, "nmrfit_pso_begin has not been called on every context");
        if (int rc = comm_stream(c, &sts[r])) return rc;
        if (int rc = stage_random(c, n_generations, rp_all ? rp_all[r] : nullptr, rg_all ? rg_all[r] : nullptr,
                                  "rp_all and rg_all", sts[r], &rp_d[r], &rg_d[r]))
            return rc;
    }
    // generation by generation over the contexts: every rank's kernels are queued before the host waits for anything
    for (int k = 0; k < n_generations; ++k) {
        for (int r = 0; r < n; ++r) {
            nmrfit_ctx* c = ctxs[r];
            CK(cudaSetDevice(c->device));
            const size_t nsd = (size_t)c->sw.B * c->sw.S * c->sw.D;
            if (int rc = queue_generations(c, 1, rp_d[r] ? rp_d[r] + nsd * k : nullptr, rg_d[r] ? rg_d[r] + nsd * k : nullptr,
                                           2, sts[r]))
                return rc;
        }
    }
    for (int r = 0; r < n; ++r) {
        CK(cudaSetDevice(ctxs[r]->device));
        if (int rc = queue_stop_flags(ctxs[r], ctxs[r]->peer_err.ptr, sts[r])) return rc;
    }
    int running = 0, lost = 0;
    for (int r = 0; r < n; ++r) {
        nmrfit_ctx* c = ctxs[r];
        CK(cudaSetDevice(c->device));
        CK(cudaStreamSynchronize(sts[r]));
        lost |= c->h_flags.ptr[c->sw.B];
        if (r == 0) running = running_spectra(c);          // identical on every rank
    }
    if (n_running) *n_running = running;
    if (timed_out) *timed_out = lost;
    return NMRFIT_OK;
}

int nmrfit_pso_peer_timeout(nmrfit_ctx* c, double milliseconds) {
    if (int rc = check_ctx(c)) return rc;
    if (!(milliseconds > 0.0)) return fail(NMRFIT_ERR_ARG, "the timeout must be positive");
    c->peer_timeout_ms = milliseconds;
    return NMRFIT_OK;
}

int nmrfit_pso_peer_error(nmrfit_ctx* c, int* timed_out) {
    if (int rc = check_ctx(c)) return rc;
    if (!timed_out) return fail(NMRFIT_ERR_ARG, "timed_out is NULL");
    *timed_out = 0;
    if (!c->peers_ready) return NMRFIT_OK;
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpy(timed_out, c->peer_err.ptr, sizeof(int), cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_pso_record(nmrfit_ctx* c, double** rec_dev, int* n_doubles) {
    if (int rc = require_swarm(c)) return rc;
    if (rec_dev) *rec_dev = c->sw.rec;
    if (n_doubles) *n_doubles = c->B * (c->D + 2);
    return NMRFIT_OK;
}

int nmrfit_pso_commit(nmrfit_ctx* c, const double* recs_dev, int n_ranks, void* stream) {
    if (int rc = require_swarm(c)) return rc;
    if (recs_dev && n_ranks < 1) return fail(NMRFIT_ERR_ARG, "n_ranks must be >= 1");
    CK(cudaSetDevice(c->device));
    const double* recs = recs_dev ? recs_dev : c->sw.rec;
    cudaError_t e = launch_swarm_commit(c->sw, recs, recs_dev ? n_ranks : 1, c->generation == 0, c->maxiter,
                                        (cudaStream_t)stream);
    if (e != cudaSuccess) return fail_cuda(e, "swarm commit");
    return NMRFIT_OK;
}

int nmrfit_pso_run(nmrfit_ctx* c, int n_generations, const double* rp_all, const double* rg_all, int* n_running,
                   void* stream) {
    if (int rc = require_swarm(c)) return rc;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const SwarmState& s = c->sw;
    const double *rp_d, *rg_d;
    if (int rc = stage_random(c, n_generations, rp_all, rg_all, "rp_all and rg_all", st, &rp_d, &rg_d)) return rc;
    FusedArgs fa;
    FusedPlan plan{};
    if (n_generations > 0)
        if (int rc = fused_setup(c, n_generations, rp_d, rg_d, &fa, &plan)) return rc;
    if (c->fused_mode == NMRFIT_FUSED_REQUIRE && n_generations > 0 && !plan.ok)
        return fail(NMRFIT_ERR_STATE, "the fused swarm kernel cannot run this shape (needs FP64, a uniform axis, the real-only "
                                      "fit and n_spectra * swarmsize CTAs co-resident)");
    if (plan.ok) {
        cudaError_t e = launch_swarm_fused(fa, plan, s.B, s.S, st);
        if (e != cudaSuccess) return fail_cuda(e, "fused swarm launch");
        c->generation += n_generations;
        c->fused_launches += 1;
        n_generations = 0;
    }
    if (int rc = queue_generations(c, n_generations, rp_d, rg_d, 1, st)) return rc;
    if (int rc = queue_stop_flags(c, c->ferror.ptr, st)) return rc;
    CK(cudaStreamSynchronize(st));
    if (c->h_flags.ptr[s.B])
        return fail(NMRFIT_ERR_STATE, "fused swarm kernel: the barrier among the CTAs of a spectrum timed out (a CTA died); "
                                      "the swarm state is undefined");
    if (n_running) *n_running = running_spectra(c);
    return NMRFIT_OK;
}

int nmrfit_pso_get_best(nmrfit_ctx* c, double* x_best, double* f_best, int* generations, int* stop_reason) {
    if (int rc = require_swarm(c)) return rc;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    const SwarmState& s = c->sw;
    if (x_best) CK(cudaMemcpy(x_best, s.best_x, sizeof(double) * s.B * s.D, cudaMemcpyDeviceToHost));
    if (f_best) CK(cudaMemcpy(f_best, s.best_f, sizeof(double) * s.B, cudaMemcpyDeviceToHost));
    if (generations) CK(cudaMemcpy(generations, s.it, sizeof(int) * s.B, cudaMemcpyDeviceToHost));
    if (stop_reason) CK(cudaMemcpy(stop_reason, s.stop, sizeof(int) * s.B, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_pso_get_state(nmrfit_ctx* c, double* x, double* v, double* p, double* fx, double* fp) {
    if (int rc = require_swarm(c)) return rc;
    CK(cudaSetDevice(c->device));
    CK(cudaDeviceSynchronize());
    const SwarmState& s = c->sw;
    size_t nsd = sizeof(double) * s.B * s.S * s.D, ns = sizeof(double) * s.B * s.S;
    if (x) CK(cudaMemcpy(x, s.x, nsd, cudaMemcpyDeviceToHost));
    if (v) CK(cudaMemcpy(v, s.v, nsd, cudaMemcpyDeviceToHost));
    if (p) CK(cudaMemcpy(p, s.p, nsd, cudaMemcpyDeviceToHost));
    if (fx) CK(cudaMemcpy(fx, s.fx, ns, cudaMemcpyDeviceToHost));
    if (fp) CK(cudaMemcpy(fp, s.fp, ns, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

// ---- curves --------------------------------------------------------------------------------------

int nmrfit_ps2(const double* u, const double* v, int n, double p0, double p1, int inv, double* re, double* im,
               void* stream) {
    if (n < 0 || (n > 0 && (!u || !v || !re || !im))) return fail(NMRFIT_ERR_ARG, "bad ps2 arguments");
    cudaError_t e = launch_ps2(u, v, n, p0, p1, inv, re, im, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail_cuda(e, "ps2 launch");
    return NMRFIT_OK;
}

int nmrfit_voigt(const double* w, int n, double r, double yoff, double width, double loc, double a, double* out,
                 void* stream) {
    if (n < 0 || (n > 0 && (!w || !out))) return fail(NMRFIT_ERR_ARG, "bad voigt arguments");
    cudaError_t e = launch_voigt(w, n, r, yoff, width, loc, a, out, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail_cuda(e, "voigt launch");
    return NMRFIT_OK;
}

int nmrfit_kk(const double* w, int n, double r, double yoff, double width, double loc, double a, double* out,
              void* stream) {
    (void)yoff;   // cancels in the Kramers-Kronig integrand (equations.py:40,45,48)
    if (n < 0 || (n > 0 && (!w || !out))) return fail(NMRFIT_ERR_ARG, "bad kk arguments");
    cudaError_t e = launch_kk(w, n, r, width, loc, a, out, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail_cuda(e, "kk launch");
    return NMRFIT_OK;
}

int nmrfit_generate_result(const double* params, int P, const double* w, int n, double* real, double* imag, double* V,
                           double* I, double* u, double* v, void* stream) {
    if (!params || P < 1 || n < 0) return fail(NMRFIT_ERR_ARG, "bad generate_result arguments");
    if (n > 0 && (!w || !real || !imag || !V || !I || !u || !v)) return fail(NMRFIT_ERR_ARG, "NULL output buffer");
    if (n == 0) return NMRFIT_OK;
    cudaError_t e = launch_generate_result(params, P, w, n, real, imag, V, I, u, v, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail_cuda(e, "generate_result launch");
    return NMRFIT_OK;
}

// host-staged variants: copy in, run, copy out.  Their device staging comes from a per-thread, per-device arena that is
// kept between calls (a cudaMalloc/cudaFree pair costs more than these kernels run); requests beyond kArenaKeep are
// served by a temporary allocation instead, so one large call does not pin device memory for good.
namespace {
constexpr size_t kArenaKeep = (size_t)8 << 20;             // doubles (64 MB)
struct Arena {
    double* ptr = nullptr;
    size_t cap = 0;
};
thread_local Arena t_arena[NMRFIT_MAX_DEVICES];

struct Scratch {
    double* base = nullptr;
    double* temp = nullptr;                                // temporary allocation of an oversized request
    size_t used = 0, total = 0;
    cudaError_t err = cudaSuccess;
    Scratch(int device, size_t total_doubles) : total(std::max<size_t>(total_doubles, 1)) {
        if (total > kArenaKeep || device < 0 || device >= NMRFIT_MAX_DEVICES) {
            err = cudaMalloc(&temp, total * sizeof(double));
            base = temp;
            return;
        }
        Arena& a = t_arena[device];
        if (a.cap < total) {
            if (a.ptr) cudaFree(a.ptr);
            a.ptr = nullptr;
            a.cap = 0;
            err = cudaMalloc(&a.ptr, total * sizeof(double));
            if (err == cudaSuccess) a.cap = total;
        }
        base = a.ptr;
    }
    ~Scratch() { if (temp) cudaFree(temp); }
    double* take(size_t n) {
        double* p = base + used;
        used += std::max<size_t>(n, 1);
        return p;
    }
};
}  // namespace

int nmrfit_ps2_host(int device, const double* u, const double* v, int n, double p0, double p1, int inv, double* re,
                    double* im) {
    if (n < 0 || (n > 0 && (!u || !v || !re || !im))) return fail(NMRFIT_ERR_ARG, "bad ps2 arguments");
    if (n == 0) return NMRFIT_OK;
    CK(cudaSetDevice(device));
    Scratch s(device, 4 * (size_t)n);
    CK(s.err);
    double *du = s.take(n), *dv = s.take(n), *dr = s.take(n), *di = s.take(n);
    CK(cudaMemcpy(du, u, sizeof(double) * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dv, v, sizeof(double) * n, cudaMemcpyHostToDevice));
    if (int rc = nmrfit_ps2(du, dv, n, p0, p1, inv, dr, di, nullptr)) return rc;
    CK(cudaMemcpy(re, dr, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(im, di, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_voigt_host(int device, const double* w, int n, double r, double yoff, double width, double loc, double a,
                      double* out) {
    if (n < 0 || (n > 0 && (!w || !out))) return fail(NMRFIT_ERR_ARG, "bad voigt arguments");
    if (n == 0) return NMRFIT_OK;
    CK(cudaSetDevice(device));
    Scratch s(device, 2 * (size_t)n);
    CK(s.err);
    double *dw = s.take(n), *dout = s.take(n);
    CK(cudaMemcpy(dw, w, sizeof(double) * n, cudaMemcpyHostToDevice));
    if (int rc = nmrfit_voigt(dw, n, r, yoff, width, loc, a, dout, nullptr)) return rc;
    CK(cudaMemcpy(out, dout, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_kk_host(int device, const double* w, int n, double r, double yoff, double width, double loc, double a,
                   double* out) {
    if (n < 0 || (n > 0 && (!w || !out))) return fail(NMRFIT_ERR_ARG, "bad kk arguments");
    if (n == 0) return NMRFIT_OK;
    CK(cudaSetDevice(device));
    Scratch s(device, 2 * (size_t)n);
    CK(s.err);
    double *dw = s.take(n), *dout = s.take(n);
    CK(cudaMemcpy(dw, w, sizeof(double) * n, cudaMemcpyHostToDevice));
    if (int rc = nmrfit_kk(dw, n, r, yoff, width, loc, a, dout, nullptr)) return rc;
    CK(cudaMemcpy(out, dout, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_generate_result_host(int device, const double* params, int P, const double* w, int n, double* real,
                                double* imag, double* V, double* I, double* u, double* v) {
    if (!params || P < 1 || n < 0) return fail(NMRFIT_ERR_ARG, "bad generate_result arguments");
    if (n > 0 && (!w || !real || !imag || !V || !I || !u || !v)) return fail(NMRFIT_ERR_ARG, "NULL output buffer");
    if (n == 0) return NMRFIT_OK;
    CK(cudaSetDevice(device));
    size_t pn = (size_t)P * n;
    Scratch s(device, 2 * pn + 5 * (size_t)n);
    CK(s.err);
    double *dw = s.take(n), *dreal = s.take(pn), *dimag = s.take(pn);
    double *dV = s.take(n), *dI = s.take(n), *du = s.take(n), *dv = s.take(n);
    CK(cudaMemcpy(dw, w, sizeof(double) * n, cudaMemcpyHostToDevice));
    if (int rc = nmrfit_generate_result(params, P, dw, n, dreal, dimag, dV, dI, du, dv, nullptr)) return rc;
    CK(cudaMemcpy(real, dreal, sizeof(double) * pn, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(imag, dimag, sizeof(double) * pn, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(V, dV, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(I, dI, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(u, du, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(v, dv, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

// ---- phase estimation ----------------------------------------------------------------------------

int nmrfit_phase_create(nmrfit_phase** out, int device, int n_spectra, int n_points, const double* u, const double* v) {
    if (!out) return fail(NMRFIT_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (n_spectra < 1 || n_points < 2 || !u || !v) return fail(NMRFIT_ERR_ARG, "bad phase arguments");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(NMRFIT_ERR_ARG, "no such CUDA device");
    CK(cudaSetDevice(device));
    std::unique_ptr<nmrfit_phase> h(new (std::nothrow) nmrfit_phase());
    if (!h) return fail(NMRFIT_ERR_NOMEM, "out of host memory");
    h->device = device; h->B = n_spectra; h->N = n_points;
    const size_t n = (size_t)n_spectra * n_points;
    CK(h->u.reserve(n));
    CK(h->v.reserve(n));
    CK(cudaMemcpy(h->u.ptr, u, sizeof(double) * n, cudaMemcpyDefault));
    CK(cudaMemcpy(h->v.ptr, v, sizeof(double) * n, cudaMemcpyDefault));
    *out = h.release();
    return NMRFIT_OK;
}

void nmrfit_phase_destroy(nmrfit_phase* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h;
}

int nmrfit_phase_brute(nmrfit_phase* h, const double* p0_candidates, int K, double* best_p0, double* best_err,
                       double* err, int* ok) {
    if (!h) return fail(NMRFIT_ERR_ARG, "handle is NULL");
    if (!p0_candidates || K < 1 || !best_p0) return fail(NMRFIT_ERR_ARG, "bad brute-phase arguments");
    CK(cudaSetDevice(h->device));
    const size_t BK = (size_t)h->B * K;
    CK(h->cands.reserve(K));
    CK(h->out.reserve(BK + 2 * (size_t)h->B));
    CK(h->ok.reserve(BK));
    CK(cudaMemcpy(h->cands.ptr, p0_candidates, sizeof(double) * K, cudaMemcpyDefault));
    double* d_best = h->out.ptr + BK;
    cudaError_t e = launch_phase_brute(h->u.ptr, h->v.ptr, h->B, h->N, h->cands.ptr, K, h->out.ptr, h->ok.ptr, d_best,
                                       d_best + h->B, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "brute phase launch");
    CK(cudaMemcpy(best_p0, d_best, sizeof(double) * h->B, cudaMemcpyDeviceToHost));
    if (best_err) CK(cudaMemcpy(best_err, d_best + h->B, sizeof(double) * h->B, cudaMemcpyDeviceToHost));
    if (err) CK(cudaMemcpy(err, h->out.ptr, sizeof(double) * BK, cudaMemcpyDeviceToHost));
    if (ok) CK(cudaMemcpy(ok, h->ok.ptr, sizeof(int) * BK, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_phase_acme(nmrfit_phase* h, const double* ph, int K, double* score) {
    if (!h) return fail(NMRFIT_ERR_ARG, "handle is NULL");
    if (!ph || K < 1 || !score) return fail(NMRFIT_ERR_ARG, "bad ACME arguments");
    CK(cudaSetDevice(h->device));
    const size_t BK = (size_t)h->B * K;
    CK(h->cands.reserve(2 * (size_t)K));
    CK(h->out.reserve(BK));
    CK(cudaMemcpy(h->cands.ptr, ph, sizeof(double) * 2 * K, cudaMemcpyDefault));
    cudaError_t e = launch_phase_acme(h->u.ptr, h->v.ptr, h->B, h->N, h->cands.ptr, K, h->out.ptr, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "ACME launch");
    CK(cudaMemcpy(score, h->out.ptr, sizeof(double) * BK, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

// ---- auto peak selection --------------------------------------------------------------------------

namespace {
// scipy.signal.savgol_coeffs(11, 4) and the degree-4 edge fits of scipy's mode='interp' (first / last 11 samples ->
// samples 0..4 / 6..10), as numpy computes them (tools/gen_sg.py); callers may pass their own
const double kSgDefault[11 + 110] = {
#include "sg_coeffs.inc"
};
}  // namespace

int nmrfit_peaks_create(nmrfit_peaks** out, int device, int n_spectra, int n_points, int upsample, int max_peaks) {
    if (!out) return fail(NMRFIT_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (n_spectra < 1 || n_points < 2 || upsample < 1 || max_peaks < 1) return fail(NMRFIT_ERR_ARG, "bad peak-selector arguments");
    if ((long long)n_points * upsample < 11) return fail(NMRFIT_ERR_ARG, "the upsampled axis needs at least 11 samples (Savitzky-Golay window)");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(NMRFIT_ERR_ARG, "no such CUDA device");
    CK(cudaSetDevice(device));
    std::unique_ptr<nmrfit_peaks> h(new (std::nothrow) nmrfit_peaks());
    if (!h) return fail(NMRFIT_ERR_NOMEM, "out of host memory");
    h->device = device; h->B = n_spectra; h->N = n_points; h->upsample = upsample; h->max_peaks = max_peaks;
    h->M = (long long)n_points * upsample;
    h->nblk = (int)((h->M + 1023) / 1024);
    const size_t BN = (size_t)n_spectra * n_points, BM = (size_t)n_spectra * h->M, BK = (size_t)n_spectra * max_peaks;
    CK(h->w.reserve(BN));
    CK(h->u.reserve(BN));
    CK(h->uu.reserve(BM));
    CK(h->us.reserve(BM));
    CK(h->bmax.reserve((size_t)n_spectra * h->nblk));
    CK(h->base.reserve(n_spectra));
    CK(h->uu_at.reserve(BK));
    CK(h->pk_h.reserve(BK));
    CK(h->sg.reserve(121));
    CK(h->maxima.reserve(BK));
    CK(h->pk_i.reserve(BK));
    CK(h->cross.reserve(2 * BK));
    CK(h->n_maxima.reserve(n_spectra));
    CK(h->n_pk.reserve(n_spectra));
    CK(h->out.reserve(BK * peaks_out_bytes()));
    *out = h.release();
    return NMRFIT_OK;
}

void nmrfit_peaks_destroy(nmrfit_peaks* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    delete h;
}

int nmrfit_peaks_maxima(nmrfit_peaks* h, const double* w, const double* u, double window, const double* sg_coeffs,
                        int baseline_max_it, double baseline_tol, int* n_maxima, long long* maxima, double* uu_at_maxima,
                        double* baseline) {
    if (!h) return fail(NMRFIT_ERR_ARG, "handle is NULL");
    if (!w || !u || !n_maxima || !maxima || !uu_at_maxima || !baseline) return fail(NMRFIT_ERR_ARG, "NULL argument");
    if (baseline_max_it < 1 || !(baseline_tol > 0.0)) return fail(NMRFIT_ERR_ARG, "bad baseline iteration arguments");
    CK(cudaSetDevice(h->device));
    const size_t BN = (size_t)h->B * h->N, BK = (size_t)h->B * h->max_peaks;
    CK(cudaMemcpy(h->w.ptr, w, sizeof(double) * BN, cudaMemcpyDefault));
    CK(cudaMemcpy(h->u.ptr, u, sizeof(double) * BN, cudaMemcpyDefault));
    // the axis must ascend (interp1d sorts; the caller mirrors that) and the window is in its units
    std::vector<double> ends(2 * (size_t)h->B);
    CK(cudaMemcpy2D(ends.data(), 2 * sizeof(double), h->w.ptr, sizeof(double) * h->N, sizeof(double), h->B, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy2D(ends.data() + 1, 2 * sizeof(double), h->w.ptr + (h->N - 1), sizeof(double) * h->N, sizeof(double), h->B,
                    cudaMemcpyDeviceToHost));
    long long order = -1;
    for (int b = 0; b < h->B; ++b) {
        const double start = ends[2 * b], stop = ends[2 * b + 1];
        if (!(stop > start)) return fail(NMRFIT_ERR_ARG, "w must be ascending (sort it as scipy's interp1d would)");
        // utils.py:728-729: x_spacing = w[1] - w[0] of the upsampled axis; window = int(window / x_spacing)
        const double step = (stop - start) / (double)(h->M - 1);
        const double w1 = h->M == 2 ? stop : 1.0 * step + start;
        const long long ob = (long long)(window / (w1 - start));
        if (order < 0) order = ob;
        else if (ob != order) return fail(NMRFIT_ERR_ARG, "every spectrum of a batch must give the same window in samples");
    }
    if (order < 1) return fail(NMRFIT_ERR_ARG, "window is shorter than one upsampled sample");      // scipy: order >= 1
    CK(cudaMemcpy(h->sg.ptr, sg_coeffs ? sg_coeffs : kSgDefault, sizeof(double) * 121, cudaMemcpyHostToDevice));
    std::vector<double> sg(121);
    std::memcpy(sg.data(), sg_coeffs ? sg_coeffs : kSgDefault, sizeof(double) * 121);
    cudaError_t e = launch_peaks_front(h->w.ptr, h->u.ptr, h->B, h->N, h->M, sg.data(), h->uu.ptr, h->us.ptr, h->bmax.ptr,
                                       h->nblk, h->base.ptr, baseline_max_it, baseline_tol, order, h->max_peaks,
                                       h->maxima.ptr, h->n_maxima.ptr, h->uu_at.ptr, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "peak-selector front launch");
    CK(cudaMemcpy(n_maxima, h->n_maxima.ptr, sizeof(int) * h->B, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(maxima, h->maxima.ptr, sizeof(long long) * BK, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(uu_at_maxima, h->uu_at.ptr, sizeof(double) * BK, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(baseline, h->base.ptr, sizeof(double) * h->B, cudaMemcpyDeviceToHost));
    for (int b = 0; b < h->B; ++b)
        if (n_maxima[b] > h->max_peaks)
            return fail(NMRFIT_ERR_STATE, "more maxima than max_peaks in spectrum " + std::to_string(b) + " (" +
                                          std::to_string(n_maxima[b]) + "): raise max_peaks or the window");
    h->ran = true;
    return NMRFIT_OK;
}

int nmrfit_peaks_measure(nmrfit_peaks* h, const int* n_peaks, const long long* peak_i, const double* peak_height,
                         int baseline_max_it, double baseline_tol, int* ok, double* loc, double* width, double* bounds,
                         double* local_baseline, double* height, double* area, long long* idx_range) {
    if (!h) return fail(NMRFIT_ERR_ARG, "handle is NULL");
    if (!h->ran) return fail(NMRFIT_ERR_STATE, "nmrfit_peaks_maxima has not been called");
    if (!n_peaks || !peak_i || !peak_height || !ok || !loc || !width || !bounds || !local_baseline || !height || !area || !idx_range)
        return fail(NMRFIT_ERR_ARG, "NULL argument");
    CK(cudaSetDevice(h->device));
    const size_t BK = (size_t)h->B * h->max_peaks;
    for (int b = 0; b < h->B; ++b)
        if (n_peaks[b] < 0 || n_peaks[b] > h->max_peaks) return fail(NMRFIT_ERR_ARG, "n_peaks out of range");
    CK(cudaMemcpy(h->n_pk.ptr, n_peaks, sizeof(int) * h->B, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->pk_i.ptr, peak_i, sizeof(long long) * BK, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->pk_h.ptr, peak_height, sizeof(double) * BK, cudaMemcpyHostToDevice));
    CK(cudaMemset(h->out.ptr, 0, BK * peaks_out_bytes()));
    cudaError_t e = launch_peaks_back(h->w.ptr, h->uu.ptr, h->B, h->N, h->M, h->base.ptr, h->pk_i.ptr, h->pk_h.ptr, h->n_pk.ptr,
                                      h->max_peaks, h->cross.ptr, baseline_max_it, baseline_tol, h->out.ptr, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "peak-selector back launch");
    struct PeakOutHost { double loc, width, b0, b1, baseline, height, area; long long lo, hi; int ok; int pad; };
    static_assert(sizeof(PeakOutHost) == 80, "PeakOut layout");
    if (peaks_out_bytes() != sizeof(PeakOutHost)) return fail(NMRFIT_ERR_STATE, "PeakOut layout mismatch");
    std::vector<PeakOutHost> res(BK);
    CK(cudaMemcpy(res.data(), h->out.ptr, BK * sizeof(PeakOutHost), cudaMemcpyDeviceToHost));
    for (size_t q = 0; q < BK; ++q) {
        ok[q] = res[q].ok; loc[q] = res[q].loc; width[q] = res[q].width; bounds[2 * q] = res[q].b0; bounds[2 * q + 1] = res[q].b1;
        local_baseline[q] = res[q].baseline; height[q] = res[q].height; area[q] = res[q].area;
        idx_range[2 * q] = res[q].lo; idx_range[2 * q + 1] = res[q].hi;
    }
    return NMRFIT_OK;
}

int nmrfit_peaks_probe(nmrfit_peaks* h, int b, const long long* idx, int n, double* wu, double* uu, double* us) {
    if (!h) return fail(NMRFIT_ERR_ARG, "handle is NULL");
    if (!h->ran) return fail(NMRFIT_ERR_STATE, "nmrfit_peaks_maxima has not been called");
    if (b < 0 || b >= h->B || n < 1 || !idx || !wu || !uu || !us) return fail(NMRFIT_ERR_ARG, "bad probe arguments");
    for (int k = 0; k < n; ++k)
        if (idx[k] < 0 || idx[k] >= h->M) return fail(NMRFIT_ERR_ARG, "probe index out of range");
    CK(cudaSetDevice(h->device));
    CK(h->probe_idx.reserve(n));
    CK(h->probe_out.reserve(3 * (size_t)n));
    CK(cudaMemcpy(h->probe_idx.ptr, idx, sizeof(long long) * n, cudaMemcpyHostToDevice));
    cudaError_t e = launch_peaks_probe(h->w.ptr, h->N, h->M, h->uu.ptr, h->us.ptr, b, h->probe_idx.ptr, n, h->probe_out.ptr, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "peak-selector probe launch");
    CK(cudaMemcpy(wu, h->probe_out.ptr, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(uu, h->probe_out.ptr + n, sizeof(double) * n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(us, h->probe_out.ptr + 2 * (size_t)n, sizeof(double) * n, cudaMemcpyDeviceToHost));
    return NMRFIT_OK;
}

int nmrfit_host_alloc(size_t bytes, void** out) {
    if (!out || bytes == 0) return fail(NMRFIT_ERR_ARG, "bad host_alloc arguments");
    *out = nullptr;
    CK(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return NMRFIT_OK;
}

int nmrfit_host_free(void* p) {
    if (!p) return NMRFIT_OK;
    CK(cudaFreeHost(p));
    return NMRFIT_OK;
}

int nmrfit_fp64_peak(int device, int iters, int repeats, double* burst, double* sustained) {
    if (!burst || !sustained || iters < 1 || repeats < 1) return fail(NMRFIT_ERR_ARG, "bad probe arguments");
    CK(cudaSetDevice(device));
    cudaError_t e = fp64_peak_probe(iters, repeats, burst, sustained, nullptr);
    if (e != cudaSuccess) return fail_cuda(e, "fp64 probe");
    return NMRFIT_OK;
}

}  // extern "C"
