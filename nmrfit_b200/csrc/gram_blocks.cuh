// Register-blocked Gram tiling shared by the normal-equations pass (K12, normal_eq.cu) and the lagged M pass (K14,
// lagged.cu): the upper triangle of each E x E matrix is cut into RB x RB blocks ("tasks"), one per thread, and a
// CTA's point groups and task slices are laid out by the plan.  Both plans are kernel parameters, so they keep their
// own structs (NormalEqPlan, LaggedPlan) and share the fields used here by name.
// The device helpers are the code both kernels had before it was factored out: their SASS is identical to that version.
#pragma once
#include <cuda_runtime.h>

namespace nmrfit {

constexpr int RB = 4;                  // register block edge

// upper-triangle block q of an nb x nb block grid -> (row block, column block), row-major over bi <= bj
__device__ __forceinline__ void tri_block(int q, int nb, int* bi, int* bj) {
    int i = 0;
    while (q >= nb - i) { q -= nb - i; ++i; }
    *bi = i;
    *bj = i + q;
}

// the inverse: the block q holding element (j, k), j <= k
__device__ __forceinline__ int tri_index(int j, int k, int nb) {
    const int bi = j / RB, bj = k / RB;
    return bi * nb - bi * (bi - 1) / 2 + (bj - bi);
}

// thread tid of task slice `slice`: its point group, its task (over all matrices) and whether it has one
template <typename Plan>
__device__ __forceinline__ void gram_task(const Plan& p, int slice, int tid, int* grp, int* task, bool* active) {
    const int task0 = slice * p.tasks_per_slice;
    *grp = p.ng > 1 ? tid / p.tasks : 0;
    *task = task0 + (p.ng > 1 ? tid - *grp * p.tasks : tid);
    *active = *grp < p.ng && *task < p.tasks && (p.ng > 1 || tid < p.tasks_per_slice);
}

__device__ __forceinline__ void gram_zero(double (&acc)[RB][RB]) {
#pragma unroll
    for (int i = 0; i < RB; ++i)
#pragma unroll
        for (int j = 0; j < RB; ++j) acc[i][j] = 0.0;
}

// End of a chunk: the point groups' blocks added in group order (through `red`, [nt][RB*RB] of shared memory), then
// one block per task to the chunk's partials out [tasks][RB*RB].  Every thread of the CTA calls it.
template <typename Plan>
__device__ __forceinline__ void gram_store(const Plan& p, const double (&acc)[RB][RB], bool active, int task, int tid,
                                           int nt, double* red, double* out) {
    if (p.ng > 1) {
        __syncthreads();
        if (active)
#pragma unroll
            for (int u = 0; u < RB; ++u)
#pragma unroll
                for (int v = 0; v < RB; ++v) red[tid * RB * RB + u * RB + v] = acc[u][v];
        __syncthreads();
        for (int idx = tid; idx < p.tasks * RB * RB; idx += nt) {
            const int tk = idx / (RB * RB), e = idx - tk * (RB * RB);
            double s = 0.0;
            for (int gi = 0; gi < p.ng; ++gi) s += red[(gi * p.tasks + tk) * RB * RB + e];
            out[idx] = s;
        }
    } else if (active) {
#pragma unroll
        for (int u = 0; u < RB; ++u)
#pragma unroll
            for (int v = 0; v < RB; ++v) out[(size_t)task * RB * RB + u * RB + v] = acc[u][v];
    }
}

// Host: the block layout of a plan for `mats` matrices of edge E (nb, ep, tasks, ng, slices, tasks_per_slice,
// threads); returns the blocks of one triangle.
template <typename Plan>
inline int gram_layout(Plan& p, int E, int mats) {
    p.nb = (E + RB - 1) / RB;
    p.ep = p.nb * RB;
    const int tri = p.nb * (p.nb + 1) / 2;
    p.tasks = mats * tri;
    if (p.tasks <= 128) {                                 // few blocks: point groups share the tile
        p.ng = 256 / p.tasks;
        p.slices = 1;
        p.tasks_per_slice = p.tasks;
        p.threads = (p.ng * p.tasks + 31) / 32 * 32;
    } else {                                              // many blocks: up to 512 per CTA, the rest in further slices
        p.ng = 1;
        p.slices = (p.tasks + 511) / 512;
        p.tasks_per_slice = (p.tasks + p.slices - 1) / p.slices;
        p.threads = (p.tasks_per_slice + 31) / 32 * 32;
    }
    return tri;
}

// Host: points per CTA for matrices of edge E, about 2^22 Gram FMAs per matrix, between 256 points and N/128 rounded up
inline int gram_chunk(int N, int E) {
    const long long target = (1LL << 22) / ((long long)E * E);
    int ch = 256;
    while ((long long)ch * 2 <= target && ch < 16384) ch *= 2;
    while ((long long)ch * 128 < N) ch *= 2;
    return ch;
}

}  // namespace nmrfit
