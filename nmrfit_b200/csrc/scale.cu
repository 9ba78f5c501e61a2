// K17: the residuals at one parameter vector per spectrum, and their median and median absolute deviation (FP64)
//
// residuals_kernel: res [B][N] with res_i from ne_residual (normal_eq_rows.cuh), the residual every post-fit pass
// sees.  CTA = (chunk of kResChunk points, spectrum), one point per thread and step; no reduction.
//
// median_mad_kernel: one CTA per spectrum finds med = median(res) and MAD = median(|res - med|) with numpy's
// semantics (the middle order statistic for odd N, (a + b) / 2 of the two middle ones for even N, NaN for a row
// holding a NaN) by an exact radix selection:
//   * each value is keyed by the order-preserving map of its bits to uint64 (-0 as +0), so that key order is value
//     order; the key sought is built a digit of 8 bits at a time from the top: a histogram of the digit over the
//     values that match the digits found so far, then the bucket holding the rank sought (8 passes);
//   * the row's keys are staged in shared memory when N <= kStageKeys; a longer row is read from global memory (and
//     L2) until the values that match the prefix fit there, then gathered once;
//   * for even N the upper middle value is the lower one again when enough values equal it, else the least key
//     above it (one more pass over the row);
//   * MAD runs the same selection on fabs(res - med), the expression numpy evaluates.
// The histogram counts are integers, so the warp-aggregated shared atomics are exact and the selected values are
// elements of the row: the result depends on nothing but the row.
#include <cuda_runtime.h>
#include <stdint.h>
#include "nmrfit_internal.h"
#include "normal_eq_rows.cuh"

namespace nmrfit {

namespace {

constexpr int kResThreads = 256;
constexpr int kResChunk = 1024;
constexpr int kSelThreads = 1024;
constexpr int kStageKeys = 24576;                     // 192 KB of keys in shared memory
constexpr int kBins = 256;
constexpr unsigned kFull = 0xffffffffu;

__global__ void __launch_bounds__(kResThreads) residuals_kernel(const double* __restrict__ spec,
                                                                const double* __restrict__ xs, int N, int P,
                                                                double* __restrict__ res) {
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.y, tid = threadIdx.x, D = 4 + 3 * P;
    const double* sw = spec + (size_t)b * 4 * N;
    const double* x = xs + (size_t)b * D;
    PeakK* pk = reinterpret_cast<PeakK*>(smem);       // [P]
    for (int k = tid; k < P; k += kResThreads) {
        PeakK c;
        ne_peak_constants(x, k, c);
        pk[k] = c;
    }
    __syncthreads();
    const double p0 = x[0], p1 = x[1], r = x[2], yoff = x[3], rN = (double)N;
    const int c0 = blockIdx.x * kResChunk, c1 = min(c0 + kResChunk, N);
    for (int pt = c0 + tid; pt < c1; pt += kResThreads) {
        double wt, rs;
        ne_residual(pk, P, p0, p1, r, yoff, pt, N, rN, sw, &wt, &rs);
        res[(size_t)b * N + pt] = rs;
    }
}

// order-preserving key of a double (-0 and +0 share the key of +0) and its inverse
__device__ __forceinline__ unsigned long long order_key(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v == 0.0 ? 0.0 : v);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ double key_value(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

struct SelState {
    unsigned hist[kBins];
    unsigned long long prefix, mask, least;           // digits found, their bits, least key above the lower middle
    unsigned k, count, n_cand;                        // rank sought among the matches, matches, keys gathered
    int nan;
};

// hist[digit] += 1 for every lane with `active`, one shared atomic per distinct digit of the warp.  Every lane of the
// warp calls it.
__device__ __forceinline__ void hist_add(unsigned* hist, bool active, unsigned digit) {
    const unsigned act = __ballot_sync(kFull, active);
    if (active) {
        const unsigned peers = __match_any_sync(act, digit);
        if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[digit], (unsigned)__popc(peers));
    }
}

// warp 0: the bucket of the digit at `shift` that holds rank s.k; s.k becomes the rank within it, s.count its size
__device__ void pick_bucket(SelState& s, int shift) {
    if (threadIdx.x >= 32) return;
    const int l = threadIdx.x;
    unsigned loc[kBins / 32], sum = 0;
#pragma unroll
    for (int j = 0; j < kBins / 32; ++j) {
        loc[j] = s.hist[l * (kBins / 32) + j];
        sum += loc[j];
    }
    unsigned incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(kFull, incl, o);
        if (l >= o) incl += t;
    }
    const unsigned k = s.k;
    unsigned below = incl - sum;
    if (below <= k && k < incl) {
        bool found = false;
#pragma unroll
        for (int j = 0; j < kBins / 32; ++j) {
            if (!found && below + loc[j] > k) {
                found = true;
                s.k = k - below;
                s.count = loc[j];
                s.prefix |= (unsigned long long)(l * (kBins / 32) + j) << shift;
                s.mask |= 0xffull << shift;
            }
            if (!found) below += loc[j];
        }
    }
}

// the value of row position i as the selection sees it: res_i, or fabs(res_i - med) for the MAD
template <bool Dev>
__device__ __forceinline__ double row_value(const double* row, int i, double med) {
    const double v = row[i];
    return Dev ? fabs(v - med) : v;
}

// The median of the N values row_value<Dev>(row, ., med), with numpy's semantics.  `cand` holds
// min(N, kStageKeys) keys; with `staged` it holds the row's keys already (Dev: those of the raw residuals).
template <bool Dev>
__device__ double select_median(const double* row, int N, double med, bool staged, unsigned long long* cand,
                                SelState& s) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        s.prefix = 0;
        s.mask = 0;
        s.k = (unsigned)(N - 1) / 2;
        s.nan = 0;
        s.least = ~0ull;
    }
    for (int j = tid; j < kBins; j += kSelThreads) s.hist[j] = 0;
    __syncthreads();
    // every value once: NaN check, top digit, and the keys staged (or, for the MAD, restaged) in shared memory
    for (int base = 0; base < N; base += kSelThreads) {
        const int i = base + tid;
        unsigned long long key = 0;
        if (i < N) {
            double v;
            if (staged && Dev)
                v = fabs(key_value(cand[i]) - med);
            else
                v = row_value<Dev>(row, i, med);
            if (v != v) s.nan = 1;
            key = order_key(v);
            if (staged) cand[i] = key;
        }
        hist_add(s.hist, i < N, (unsigned)(key >> 56));
    }
    __syncthreads();
    if (s.nan) return __longlong_as_double(0x7ff8000000000000ll);
    pick_bucket(s, 56);
    __syncthreads();
    bool in_smem = staged;
    int n = N;
    for (int shift = 48; shift >= 0; shift -= 8) {
        if (!in_smem && s.count <= (unsigned)kStageKeys) {
            // gather the keys that match the prefix; their order does not matter to the selection
            const unsigned long long prefix = s.prefix, mask = s.mask;
            if (tid == 0) s.n_cand = 0;
            __syncthreads();
            for (int base = 0; base < N; base += kSelThreads) {
                const int i = base + tid;
                unsigned long long key = 0;
                if (i < N) key = order_key(row_value<Dev>(row, i, med));
                const bool hit = i < N && (key & mask) == prefix;
                const unsigned hits = __ballot_sync(kFull, hit);
                unsigned at = 0;
                if ((tid & 31) == 0 && hits) at = atomicAdd(&s.n_cand, (unsigned)__popc(hits));
                at = __shfl_sync(kFull, at, 0);
                if (hit) cand[at + __popc(hits & ((1u << (tid & 31)) - 1))] = key;
            }
            __syncthreads();
            in_smem = true;
            n = (int)s.n_cand;
        }
        const unsigned long long prefix = s.prefix, mask = s.mask;
        for (int j = tid; j < kBins; j += kSelThreads) s.hist[j] = 0;
        __syncthreads();
        for (int base = 0; base < n; base += kSelThreads) {
            const int i = base + tid;
            unsigned long long key = 0;
            if (i < n) key = in_smem ? cand[i] : order_key(row_value<Dev>(row, i, med));
            hist_add(s.hist, i < n && (key & mask) == prefix, (unsigned)(key >> shift) & 0xffu);
        }
        __syncthreads();
        pick_bucket(s, shift);
        __syncthreads();
    }
    const unsigned long long lo_key = s.prefix;
    const double lo = key_value(lo_key);
    if (N & 1) return lo;
    if (s.k + 1 < s.count) return (lo + lo) / 2.0;
    // the upper middle value is the least key above the lower one, over the whole row
    unsigned long long least = ~0ull;
    for (int i = tid; i < N; i += kSelThreads) {
        const unsigned long long key = staged ? cand[i] : order_key(row_value<Dev>(row, i, med));
        if (key > lo_key && key < least) least = key;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) least = min(least, __shfl_xor_sync(kFull, least, o));
    if ((tid & 31) == 0) atomicMin(&s.least, least);
    __syncthreads();
    return (lo + key_value(s.least)) / 2.0;
}

__global__ void __launch_bounds__(kSelThreads, 1) median_mad_kernel(const double* __restrict__ res, int N,
                                                                 double* __restrict__ out) {
    extern __shared__ __align__(16) unsigned long long cand[];   // [min(N, kStageKeys)]
    __shared__ SelState s;
    const int b = blockIdx.x;
    const double* row = res + (size_t)b * N;
    const bool staged = N <= kStageKeys;
    const double med = select_median<false>(row, N, 0.0, staged, cand, s);
    __syncthreads();
    const double mad = med != med ? med : select_median<true>(row, N, med, staged, cand, s);
    if (threadIdx.x == 0) {
        out[2 * (size_t)b] = med;
        out[2 * (size_t)b + 1] = mad;
    }
}

}  // namespace

cudaError_t launch_residuals(const double* spec, const double* x, int B, int N, int P, double* res, cudaStream_t st) {
    residuals_kernel<<<dim3((N + kResChunk - 1) / kResChunk, B), kResThreads, sizeof(PeakK) * P, st>>>(spec, x, N, P,
                                                                                                     res);
    count_launches(1);
    return cudaGetLastError();
}

cudaError_t launch_median_mad(const double* res, int B, int N, double* out, cudaStream_t st) {
    const int smem = (int)sizeof(unsigned long long) * (N < kStageKeys ? N : kStageKeys);
    cudaError_t e = opt_in_smem<median_mad_kernel>((int)sizeof(unsigned long long) * kStageKeys);
    if (e != cudaSuccess) return e;
    median_mad_kernel<<<B, kSelThreads, smem, st>>>(res, N, out);
    count_launches(1);
    return cudaGetLastError();
}

}  // namespace nmrfit
