// Resident CTAs per SM of the two k_emit_lines instantiations at the shared memory they are launched with.
//   nvcc -gencode arch=compute_100a,code=sm_100a -std=c++17 -o emit_occupancy tools/emit_occupancy.cu
#include "../cactus-gfa-tools_b200/csrc/g2p_short.cuh"
#include <cstdio>

int main() {
    using namespace g2p;
    cudaFuncSetAttribute(k_emit_lines<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmitSmemMap);
    cudaFuncSetAttribute(k_emit_lines<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmitSmem);
    int n0 = 0, n1 = 0;
    cudaFuncAttributes f0, f1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n0, k_emit_lines<false>, kEThreads, kEmitSmemMap) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n1, k_emit_lines<true>, kEThreads, kEmitSmem) != cudaSuccess ||
        cudaFuncGetAttributes(&f0, k_emit_lines<false>) != cudaSuccess || cudaFuncGetAttributes(&f1, k_emit_lines<true>) != cudaSuccess) {
        std::printf("occupancy query failed\n");
        return 1;
    }
    std::printf("k_emit_lines<false>: %d regs, %zu B dynamic smem, %d CTAs/SM (%d warps)\n", f0.numRegs, kEmitSmemMap, n0, n0 * kEThreads / 32);
    std::printf("k_emit_lines<true>:  %d regs, %zu B dynamic smem, %d CTAs/SM (%d warps)\n", f1.numRegs, kEmitSmem, n1, n1 * kEThreads / 32);
    return 0;
}
