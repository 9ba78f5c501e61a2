// Resident CTAs per SM of the streamed evaluation kernel at the headline shape (6 peaks, 4,096 points: 256 threads,
// R = 8, four far-field cells per region), around the two-CTA shared-memory budget of objective_plan
// (objective_plan.h): two stages of 7 and of 8 particles, the budget itself and one byte over it.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o stream_occupancy_probe stream_occupancy_probe.cu
#include "../../nmrfit_b200/csrc/objective_stream.cu"
#include <cstdio>

int main() {
    using namespace nmrfit;
    auto k = objective_stream_kernel<256, 8, 6, 0, 2, 4>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    printf("set attr: %s\n", cudaGetErrorString(e));
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, k);
    printf("regs %d local %zu static smem %zu\n", fa.numRegs, fa.localSizeBytes, fa.sharedSizeBytes);
    int per_sm = 0, reserved = 0;
    cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, 0);
    cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, 0);
    printf("smem per SM %d, reserved per block %d\n", per_sm, reserved);
    for (int bytes : {106848, 114720, 115712, 115713}) {
        int n = -1;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, 256, bytes);
        printf("objective_stream_kernel<256,8,6,0,2,4> dynamic smem %d B: %d CTAs/SM (%s)\n", bytes, n, cudaGetErrorString(e));
    }
    return 0;
}
