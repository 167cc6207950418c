// direct_layout.cuh -- where admm_direct_kernel keeps each array of its per-instance state.  carve
// (admm_direct_kernel.cuh) lays the arrays out by this rule on the device and plan_launch (ocp_b200.cu)
// sizes the dynamic shared memory and the slab by it on the host: were the two to disagree, the kernel
// would carve past the end of one of them.
#pragma once

#include "admm_common.cuh"

namespace ocpb200 {
namespace direct {

// Placement of the per-instance state:
//   PLACE_MIXED  run-time mask (host plan: shared memory first, in kMixedPriority order; rest in a global slab)
//   PLACE_SMEM   everything in shared memory, one CTA per SM (pointers are shared-space: LDS/STS)
//   PLACE_MULTI  vectors, A values and small scratch in shared memory, factor blocks / index
//                arrays / rarely used vectors in global memory (L2-resident): ~65 KB per CTA, so that
//                three CTAs share an SM and hide each other's dependent-latency chains
//   PLACE_BIG    one CTA per SM for problems whose factor does not fit: vectors, A values, scratch and
//                index arrays in shared memory, factor blocks and set-up / check vectors in global memory
enum Placement { PLACE_MIXED = 0, PLACE_SMEM = 1, PLACE_MULTI = 2, PLACE_BIG = 3 };

// arrays of the per-instance state, in the order carve lays them out
enum ArrayId {
  AR_X = 0, AR_Q, AR_B, AR_Z, AR_Y, AR_L, AR_U, AR_CTYPE, AR_W, AR_AVAL, AR_SCRATCH, AR_STAGE, AR_IDX, AR_DINV, AR_LSUB,
  AR_PVAL, AR_LP, AR_D, AR_E, AR_DX, AR_DY, AR_COUNT
};
// AR_STAGE: two pairs of block buffers in which the factorisation stages the blocks it multiplies
// when the factor itself lives in the global slab; not allocated when everything is in shared memory.

// mixed placement: shared memory goes first to what is accessed at random or sits on the sequential path
// (solve vector, x, w, the block ring, the border scratch); vectors that are only streamed row by row (z, y,
// l, u) and the matrices follow while space lasts
constexpr int kMixedPriority[AR_COUNT] = {AR_B, AR_X, AR_W, AR_CTYPE, AR_Q, AR_STAGE, AR_SCRATCH, AR_Z, AR_Y, AR_L, AR_U,
                                          AR_D, AR_E, AR_AVAL, AR_IDX, AR_PVAL, AR_LP, AR_DINV, AR_LSUB, AR_DX, AR_DY};

__host__ __device__ inline size_t array_doubles_nominal(const PatternDev& P, int id);
__host__ __device__ inline size_t array_doubles(const PatternDev& P, int id) {
  const size_t sz = array_doubles_nominal(P, id);
  return sz > 0 ? ((sz + 1) & ~size_t(1)) + kCanaryDoubles : 0;   // guard doubles behind every array (0 unless OCP_B200_CANARY)
}
__host__ __device__ inline size_t array_doubles_nominal(const PatternDev& P, int id) {
  const size_t n = P.n, m = P.m, bs = P.tri_bs, ld = P.tri_ld, nb = P.tri_nb, np = P.tri_np;
  switch (id) {
    case AR_X: case AR_Q: case AR_B: case AR_D: case AR_DX: return (n + 1) & ~size_t(1);
    case AR_Z: case AR_Y: case AR_L: case AR_U: case AR_E: case AR_DY: return (m + 1) & ~size_t(1);
#ifdef OCP_B200_CANARY_SELFTEST   // negative control of the guard check: the round-2 bug (w sized m, written up to n) on purpose
    case AR_W: return (m + 1) & ~size_t(1);
#else
    case AR_W: return ((m > n ? m : n) + 1) & ~size_t(1);   // also the Ruiz scratch of the n column norms (QP-only handles may have m < n)
#endif
    case AR_CTYPE: return (m + 7) / 8;
    case AR_AVAL: return (size_t(P.nnz_a) + 1) & ~size_t(1);
    case AR_PVAL: return (size_t(P.nnz_p) + 1) & ~size_t(1);
    case AR_DINV: case AR_LSUB: return nb * bs * ld;
    case AR_IDX: return (size_t(P.idx_entries) * sizeof(idx_t) + 7) / 8;
    case AR_STAGE: return size_t(P.stage_slots > 0 ? P.stage_slots : 4) * ((bs * ld + 1) & ~size_t(1));
    case AR_LP: return (np * nb * bs + 1) & ~size_t(1);
    case AR_SCRATCH: return 3 * np * (np + 1) + 2 * ((bs * ld + 1) & ~size_t(1)) + 2 * ((np * bs + 1) & ~size_t(1)) +
                            ((np + 2) & ~size_t(1)) + 64;
    default: return 0;
  }
}

// the arrays a compile-time placement keeps in shared memory (bit id of ArrayId); PLACE_MIXED takes its mask from the plan
__host__ __device__ constexpr uint32_t placement_mask(int place) {
  switch (place) {
    // latency plan: everything in shared memory except the block staging buffers (not needed) and dx, which only the
    // termination checks touch -- with it the H = 20 quadrotor is 1.7 KB over the 227 KB of an SM
    case PLACE_SMEM: return ((1u << AR_COUNT) - 1u) & ~(1u << AR_STAGE | 1u << AR_DX);
    // throughput plan: vectors, A values, scratch, block staging buffers, index arrays + the small set-up / scaling
    // vectors in shared memory (109 KB for the quadrotor, two CTAs per SM); the factor blocks and dx, dy (read at
    // termination checks only) in the global slab
    case PLACE_MULTI: return ((2u << AR_IDX) - 1u) | 1u << AR_PVAL | 1u << AR_D | 1u << AR_E;
    case PLACE_BIG: return (2u << AR_IDX) - 1u;
    default: return 0u;
  }
}

// doubles of an array's slot (even, so that every slot starts 16-byte aligned); the all-shared-memory placement
// allocates no staging buffers.  array_doubles is even already and the rounding changes no value, but nvcc does not
// see that: without it the direct kernels compile to different code (16-32 bytes less stack), not measured yet.
__host__ __device__ inline size_t slot_doubles(const PatternDev& P, int place, int id) {
  return place == PLACE_SMEM && id == AR_STAGE ? 0 : (array_doubles(P, id) + 1) & ~size_t(1);
}

struct StateLayout {
  uint32_t mask;         // arrays in shared memory
  size_t smem_doubles;   // dynamic shared memory per CTA
  size_t slab_doubles;   // per-CTA global slab, rounded up to 16 doubles
};

// The host side of carve: the per-CTA sizes of the state under a placement.  PLACE_MIXED fills `avail_doubles` of
// shared memory in kMixedPriority order; force_stream keeps its factor blocks in the slab even when they would fit
// (OCP_B200_FORCE_STREAM: tests of the streamed solve on small problems).
inline StateLayout plan_state(const PatternDev& P, int place, size_t avail_doubles, bool force_stream) {
  constexpr uint32_t factor = 1u << AR_DINV | 1u << AR_LSUB | 1u << AR_LP;
  StateLayout L{placement_mask(place), 0, 0};
  for (int id : kMixedPriority) {
    const size_t sz = slot_doubles(P, place, id);
    if (place == PLACE_MIXED && !(force_stream && (factor >> id & 1u)) && L.smem_doubles + sz <= avail_doubles)
      L.mask |= 1u << id;
    (L.mask >> id & 1u ? L.smem_doubles : L.slab_doubles) += sz;
  }
  L.slab_doubles = (L.slab_doubles + 15) & ~size_t(15);
  return L;
}

}  // namespace direct
}  // namespace ocpb200
