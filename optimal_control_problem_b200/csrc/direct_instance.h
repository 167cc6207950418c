// direct_instance.h -- the host entry points of one instantiation admm_direct_kernel<kPlace, kThreads, kBlocksPerSm>.
// Each placement instantiates them in its own translation unit (direct_<placement>.cu): the kernel is large, and nvcc
// builds the units in parallel.
#pragma once
#include "admm_direct_kernel.cuh"
#include "direct_launch.h"

namespace ocpb200 {
namespace direct {

template <int kPlace, int kThreads, int kBlocksPerSm>
struct Instance {
  static cudaError_t kernel_info(KernelInfo* out) {
    cudaFuncAttributes fa{};
    cudaError_t e = cudaFuncGetAttributes(&fa, admm_direct_kernel<kPlace, kThreads, kBlocksPerSm>);
    if (e == cudaSuccess) { out->static_smem = static_cast<int>(fa.sharedSizeBytes); out->regs = fa.numRegs; out->threads = kThreads; }
    return e;
  }
  static cudaError_t set_max_dynamic_smem(int bytes) {
    return cudaFuncSetAttribute(admm_direct_kernel<kPlace, kThreads, kBlocksPerSm>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                bytes);
  }
  static cudaError_t occupancy(int dyn_smem, int* per_sm) {
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, admm_direct_kernel<kPlace, kThreads, kBlocksPerSm>, kThreads,
                                                         dyn_smem);
  }
  static cudaError_t launch(int grid, int dyn_smem, cudaStream_t st, const PatternDev& P, const ocp_b200_settings& S,
                            const SolveArgs& A, uint32_t smem_mask) {
    admm_direct_kernel<kPlace, kThreads, kBlocksPerSm><<<grid, kThreads, dyn_smem, st>>>(P, S, A, smem_mask);
    return cudaGetLastError();
  }
  static constexpr EntryPoints entry_points{&kernel_info, &set_max_dynamic_smem, &occupancy, &launch};
};

}  // namespace direct
}  // namespace ocpb200
