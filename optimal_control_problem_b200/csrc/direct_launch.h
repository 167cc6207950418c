// direct_launch.h -- host-side entry points of the instantiations of admm_direct_kernel, each
// compiled in its own translation unit (they are large; nvcc builds them in parallel).
#pragma once
#include <vector>

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

// plan helpers (host)
size_t plan_array_doubles(const PatternDev& P, int id);
int plan_array_count();
bool plan_multi_in_smem(int id);
bool plan_big_in_smem(int id);
bool plan_smem_in_smem(int id);   // latency plan (PLACE_SMEM); the rest goes to the slab
int plan_stage_array();
void plan_mixed_priority(std::vector<int>& order);
bool plan_is_factor_array(int id);   // D^-1, L, L_p blocks   // array ids, most deserving of shared memory first

}  // namespace direct
}  // namespace ocpb200
