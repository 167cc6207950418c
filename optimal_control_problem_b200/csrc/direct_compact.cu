// Instantiations of compact::admm_compact_kernel<BS, 128, 4> (admm_compact_kernel.cuh): the throughput plan for
// OCP-shaped QPs that are small enough for four CTAs per SM.
#include "admm_compact_kernel.cuh"
#include "compact_launch.h"

namespace ocpb200 {
namespace compact {

using KernelFn = void (*)(PatternDev, CompactIdx, ocp_b200_settings, SolveArgs, int);

static KernelFn kernel(int bs) {
  return bs == 16 ? admm_compact_kernel<16, kCtaThreads, kCtasPerSm> : admm_compact_kernel<20, kCtaThreads, kCtasPerSm>;
}

cudaError_t kernel_info(int bs, direct::KernelInfo* out) {
  cudaFuncAttributes fa{};
  cudaError_t e = cudaFuncGetAttributes(&fa, kernel(bs));
  if (e == cudaSuccess) { out->static_smem = static_cast<int>(fa.sharedSizeBytes); out->regs = fa.numRegs; out->threads = kCtaThreads; }
  return e;
}
cudaError_t set_max_dynamic_smem(int bs, int bytes) {
  return cudaFuncSetAttribute(kernel(bs), cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
cudaError_t launch(int bs, int grid, int dyn_smem, cudaStream_t st, const PatternDev& P, const CompactIdx& C,
                   const ocp_b200_settings& S, const SolveArgs& A, int layout_flags) {
  kernel(bs)<<<grid, kCtaThreads, dyn_smem, st>>>(P, C, S, A, layout_flags);
  return cudaGetLastError();
}
void plan_sizes(const PatternDev& P, int arena_words, int layout_flags, size_t* smem_doubles, size_t* slab_doubles, bool* ok) {
  const Layout L = make_layout(P, arena_words, layout_flags);
  *smem_doubles = L.smem_doubles; *slab_doubles = L.slab_doubles; *ok = L.ok;
}

}  // namespace compact
}  // namespace ocpb200
