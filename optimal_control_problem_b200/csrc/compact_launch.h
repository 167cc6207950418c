// compact_launch.h -- host-side entry points of the compact throughput kernel (direct_compact.cu).
#pragma once
#include "admm_common.cuh"
#include "direct_launch.h"
#include "periodic_index.h"

namespace ocpb200 {
namespace compact {

// the one shape, for block sizes 16 and 20: 128 threads x 4 CTAs/SM.  Measured on a B200, H = 20 quadrotor, sweep
// blocks in Tensor Memory: 8.55 ms per launch, against 8.84 ms at 192 threads x 3 CTAs/SM
// (profiles/r2_probe_tmem_shapes.txt).
constexpr int kCtaThreads = 128, kCtasPerSm = 4;

// layout_flags: compact::kQInSmem | kLuInSmem
cudaError_t kernel_info(int bs, direct::KernelInfo* out);
cudaError_t set_max_dynamic_smem(int bs, int bytes);
cudaError_t launch(int bs, int grid, int dyn_smem, cudaStream_t st, const PatternDev& P, const CompactIdx& C,
                   const ocp_b200_settings& S, const SolveArgs& A, int layout_flags);
void plan_sizes(const PatternDev& P, int arena_words, int layout_flags, size_t* smem_doubles, size_t* slab_doubles, bool* ok);

}  // namespace compact
}  // namespace ocpb200
