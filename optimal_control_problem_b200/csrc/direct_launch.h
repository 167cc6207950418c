// direct_launch.h -- host-side entry points of the instantiations of admm_direct_kernel, each
// compiled in its own translation unit (they are large; nvcc builds them in parallel).
#pragma once

#include "admm_common.cuh"

namespace ocpb200 {
namespace direct {

struct KernelInfo { int static_smem; int regs; int threads; };

// the host entry points of one instantiation (direct_instance.h)
struct EntryPoints {
  cudaError_t (*kernel_info)(KernelInfo* out);
  cudaError_t (*set_max_dynamic_smem)(int bytes);
  cudaError_t (*occupancy)(int dyn_smem, int* per_sm);
  cudaError_t (*launch)(int grid, int dyn_smem, cudaStream_t st, const PatternDev& P, const ocp_b200_settings& S,
                        const SolveArgs& A, uint32_t smem_mask);
};
// one instantiation per placement: direct_mixed.cu, direct_smem.cu, direct_multi.cu, direct_big.cu
extern const EntryPoints kMixed, kSmem, kMulti, kBig;

// place: 0 = mixed placement (run-time mask), 1 = all shared memory, 2 = multi-CTA-per-SM split, 3 = big problems
const EntryPoints& entry_points(int place);

}  // namespace direct
}  // namespace ocpb200
