// admm_compact_kernel.cuh -- the throughput kernel of the batched ADMM QP solve for sm_100a:
// FOUR CTAs per SM, 128 threads each.
//
// Same algorithm, same arithmetic order and the same factorisation / solve code (tri_fast.cuh,
// tri_twisted.cuh) as admm_direct_kernel.cuh -- OSQP set-up + ADMM + SQP update of B independent QPs,
// src/sqp_solver/CuCaQP.cpp:271-288, 183-224 and SQPOptimizationSolver.cpp:171-177 of the reference --
// with a different placement of the per-instance state.  The kernel is bound by dependent-instruction
// latency, not by bandwidth (DESIGN.md 5.2): what raises throughput is the number of instances an SM
// works on at the same time (profiles/r2_probe_occupancy.txt: 1 -> 2 -> 3 -> 4 CTAs/SM scale 1 : 1.73 :
// 2.29 : 2.94), and what limits that number is shared memory.  Per CTA here (H = 20 quadrotor: 50 KB,
// against 109 KB of the two-CTA plan):
//   * gather targets (solve vector b, x, w = rho z - y), the row-streamed z, y, the constraint types and
//     the A values stay in shared memory;
//   * index arrays are stage-periodic templates (periodic_index.h): 5 KB instead of 22 KB;
//   * everything that is read once per phase by the thread that owns the element -- q, l, u, D, E, the
//     P values, the Ruiz by-products -- lives in the CTA's global slab next to the factor (L2-resident)
//     and is streamed, one coalesced access per element;
//   * buffers are shared by phase: the Ruiz scratch (column / row scales, P values) and the scratch of
//     the factorisation (block staging, chain-step products) overlay the iteration vectors, which hold
//     nothing before the cold start; a refactorisation after a rho update parks x, z, y in the slab.
#pragma once

#include "admm_direct_kernel.cuh"
#include "periodic_index.h"

namespace ocpb200 {
namespace compact {

using direct::Rho;
using direct::Work;

// shared memory and slab layout (doubles); the same function runs on the host (plan) and on the device (carve)
constexpr int kMaxGuards = 40;
struct Layout {
  // guard doubles behind every array (OCP_B200_CANARY builds): offsets, and whether they lie in the slab
  int nguard;
  size_t guard_off[kMaxGuards];
  bool guard_slab[kMaxGuards];
  // shared
  size_t b, x, w, z, y, vend;       // iteration vectors; [b, vend) is also the set-up / factorisation scratch
  size_t aval, ctype, dp, xp, piv, arena, smem_doubles;
  // overlays of [b, vend)
  size_t rscale, psm;               // Ruiz: row scales on x|w, P values on z|y   (column scales are b itself)
  size_t dp2, s, sp, stage, fb;     // factorisation scratch (fb: the L_p tiles of the chain steps)
  int s_stride, sp_stride, stage_stride;
  // slab
  size_t dinv, lsub, lp, q, l, u, D, E, pval, dx, dy, an, cn, sx, sz, sy, slab_doubles;
  bool ok, q_smem, lu_smem;
};

// flags: bit 0 = q in shared memory, bit 1 = l and u in shared memory (otherwise streamed from the slab).  The scaling
// vectors D, E and the Ruiz by-products stay in the slab: in shared memory as well they made the kernel slower (H = 20
// quadrotor: 9.6 -> 9.9 ms per launch; the 10 KB are worth more as L1).
constexpr int kQInSmem = 1, kLuInSmem = 2;
__host__ __device__ inline Layout make_layout(const PatternDev& P, int arena_words, int flags) {
  auto ev = [](size_t v) { return (v + 1) & ~size_t(1); };
  const size_t n = ev(P.n), m = ev(P.m), np = P.tri_np, bs = P.tri_bs, ld = P.tri_ld, nb = P.tri_nb;
  Layout L{};
  size_t o = 0;
  auto guard = [&L](size_t& off, bool slab) {
    if (kCanaryDoubles > 0 && L.nguard < kMaxGuards) { L.guard_off[L.nguard] = off; L.guard_slab[L.nguard] = slab; ++L.nguard; off += kCanaryDoubles; }
  };
  L.b = o; o += n; L.x = o; o += n; L.w = o; o += m; L.z = o; o += m; L.y = o; o += m;
  const size_t vlen = o;
  L.s_stride = static_cast<int>(ev(bs * ld)); L.sp_stride = static_cast<int>(ev(np * bs)); L.stage_stride = L.s_stride;
  size_t f = 0;
  L.dp2 = f; f += ev(2 * np * (np + 1));
  L.s = f; f += 2 * size_t(L.s_stride);
  L.sp = f; f += 2 * size_t(L.sp_stride);
  L.stage = f; f += 4 * size_t(L.stage_stride);
  L.fb = f; f += 2 * size_t(L.sp_stride);
  L.vend = f > vlen ? f : vlen;
  o = L.vend;
  guard(o, false);
  L.rscale = L.x;   // m doubles on x|w
  L.psm = L.z;      // nnz_p doubles on z|y
  L.ok = ev(P.nnz_p) <= 2 * m && m <= n + m;
  L.aval = o; o += ev(P.nnz_a); guard(o, false);
  L.ctype = o; o += ev((size_t(P.m) + 7) / 8); guard(o, false);
  L.dp = o; o += ev(np * (np + 1)); guard(o, false);
  L.xp = o; o += ev(np + 2); guard(o, false);
  L.piv = o; o += 64; guard(o, false);
  L.arena = o; o += ev((size_t(arena_words) + 1) / 2); guard(o, false);
  size_t qs = 0, ls = 0, us = 0;
  if (flags & kQInSmem) { qs = o; o += n; guard(o, false); }
  if (flags & kLuInSmem) { ls = o; o += m; guard(o, false); us = o; o += m; guard(o, false); }
  L.smem_doubles = o;
  size_t g = 0;
  L.dinv = g; g += nb * bs * ld; guard(g, true); L.lsub = g; g += nb * bs * ld; guard(g, true); L.lp = g; g += ev(np * nb * bs); guard(g, true);
  L.q_smem = (flags & kQInSmem) != 0; L.lu_smem = (flags & kLuInSmem) != 0;
  if (L.q_smem) L.q = qs; else { L.q = g; g += n; guard(g, true); }
  if (L.lu_smem) { L.l = ls; L.u = us; } else { L.l = g; g += m; guard(g, true); L.u = g; g += m; guard(g, true); }
  L.pval = g; g += ev(P.nnz_p); guard(g, true); L.dx = g; g += n; guard(g, true); L.dy = g; g += m; guard(g, true);
  L.D = g; g += n; guard(g, true); L.E = g; g += m; guard(g, true); L.an = g; g += n; guard(g, true); L.cn = g; g += n; guard(g, true);
  // parking space of a refactorisation: dx, dy and the Ruiz by-products are dead at that point
  L.sx = L.dx; L.sz = L.dy;
  if (kCanaryDoubles == 0 && 2 * n >= m) L.sy = L.an;   // (an | cn are contiguous without guards)
   else { L.sy = g; g += m; guard(g, true); }
  L.slab_doubles = (g + 15) & ~size_t(15);
  return L;
}

struct Ctx {
  const uint32_t* ar;   // arena in shared memory
  double *rscale, *psm; // Ruiz overlays
  double *an, *cn, *sx, *sz, *sy;   // slab: Ruiz by-products, parking space of a refactorisation
  double* pslab;        // slab copy of the scaled P values
};

// (v may be a slab array written earlier in the launch by other threads of the CTA: no __restrict__)
__device__ __forceinline__ double col_dot_A(const CompactIdx& C, const uint32_t* ar, const double* __restrict__ Aval,
                                            const double* v, int j) {
  const PSpan s = pspan_dev(C.acol, ar, j);
  const uint32_t* te = ar + C.acol.tent_off;
  const double* av = Aval + s.kshift;
  double acc = 0.0;
#pragma unroll 4
  for (int kt = s.kt0; kt < s.kt1; ++kt) acc += av[kt] * v[pvalue(te[kt], s.q)];
  return acc;
}
__device__ __forceinline__ double col_dot_P(const CompactIdx& C, const uint32_t* ar, const double* Pval,
                                            const double* v, int j) {
  const PSpan s = pspan_dev(C.pcol, ar, j);
  const uint32_t* te = ar + C.pcol.tent_off;
  const double* pv = Pval + s.kshift;
  double acc = 0.0;
#pragma unroll 4
  for (int kt = s.kt0; kt < s.kt1; ++kt) acc += pv[kt] * v[pvalue(te[kt], s.q)];
  return acc;
}
// f(row, sum_k A[row][k] * src[k]) for every row, one thread per row
template <typename F>
__device__ __forceinline__ void for_rows_A(const CompactIdx& C, const uint32_t* ar, int m, const double* __restrict__ Aval,
                                           const double* src, F f) {
  const uint32_t* tc = ar + C.arow.tent_off;
  const uint32_t* tp = ar + C.arow.tent2_off;
  for (int i = threadIdx.x; i < m; i += blockDim.x) {
    const PSpan s = pspan_dev(C.arow, ar, i);
    double acc = 0.0;
    if (s.qd >= 0 && s.qd2 >= 0) {   // every entry of the row's region moves by the same delta: one 16-bit load + add
      const double* av = Aval + s.qd2;
      const double* sv = src + s.qd;
#pragma unroll 4
      for (int kt = s.kt0; kt < s.kt1; ++kt) acc += av[plow(tp, kt)] * sv[plow(tc, kt)];
    } else {
#pragma unroll 4
      for (int kt = s.kt0; kt < s.kt1; ++kt) acc += Aval[pvalue(tp[kt], s.q)] * src[pvalue(tc[kt], s.q)];
    }
    f(i, acc);
  }
}

// the sparse products of the OSQP layer (admm_common.cuh) over the templates and the arena
struct CompactOps {
  const CompactIdx& C;
  const uint32_t* ar;
  int m;
  template <typename F>
  __device__ __forceinline__ void for_rows_A(const double* Aval, const double* src, F f) const { compact::for_rows_A(C, ar, m, Aval, src, f); }
  __device__ __forceinline__ double col_dot_A(const double* Aval, const double* v, int j) const { return compact::col_dot_A(C, ar, Aval, v, j); }
  __device__ __forceinline__ double col_dot_P(const double* Pval, const double* v, int j) const { return compact::col_dot_P(C, ar, Pval, v, j); }
};

// ---------------------------------------------------------------------------------------
// Tensor Memory as the home of the sweep blocks (BS = 16).
//
// The two sweeps of a solve are the sequential critical path, and with the factor in the L2 slab every stage
// waits for a block row requested two stages earlier: ~900 cycles per stage at three CTAs per SM against ~200 in
// isolation (profiles/r2_fine_phases.txt).  Shared memory is full -- but every SM also has 256 KB of Tensor Memory
// that this FP64 path does not otherwise touch.  Each CTA allocates 128 columns (64 KB; 3-4 CTAs per SM fit into
// the 512 columns) and keeps the sub-diagonal blocks there IN THE REGISTER LAYOUT OF THE SWEEP: a block is 16
// columns, lane (row, half) of the owning warp holds its 8 doubles as 16 32-bit words, so one
// tcgen05.ld.32x32b.x16 (latency ~ a shared-memory load, tools/micro/tmem_roundtrip.cu) delivers exactly the
// operand of a stage.  A warp reaches only its own lane quadrant, so the four sweep chains go to four warps:
//   warp 0  forward, top chain     slots 1 .. mid (row layout)         + the joining slot mid + 1
//   warp 1  forward, bottom chain  slots nb-1 .. mid+2 (row layout)
//   warp 2  backward, top chain    slots mid .. 1 (column layout)
//   warp 3  backward, bottom chain slots mid+1 .. nb-1 (column layout)
// A quadrant holds 8 blocks; the last (at most 3) stages of a chain are fetched from the slab into registers when
// the sweep starts, so their latency hides behind the Tensor-Memory-fed stages.  The blocks are copied from the
// slab after every factorisation (once per QP, or per rho update).
// ---------------------------------------------------------------------------------------
constexpr int kTmemCols = 128;          // per CTA; power of two
constexpr int kTmemBlocks = kTmemCols / 16;

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const double (&d)[8]) {
  uint32_t v[16];
#pragma unroll
  for (int c = 0; c < 8; ++c) { v[2 * c] = __double2loint(d[c]); v[2 * c + 1] = __double2hiint(d[c]); }
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
                 "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, double (&d)[8]) {
  uint32_t v[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                 "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int c = 0; c < 8; ++c) d[c] = __hiloint2double(static_cast<int>(v[2 * c + 1]), static_cast<int>(v[2 * c]));
}
// (requesting the block of stage i + 1 before stage i is computed -- two register sets, the wait naming them as
//  operands -- was measured: 8.8 -> 11.8 ms per launch at 96 registers; the load is as fast as a shared-memory one)

// the chain of sweep stages one of the four sweep warps runs: stage i uses slot slot0 + i * dslot
struct SweepChain { int slot0, dslot, dst0, src0, dblk, count; bool column; };
__device__ __forceinline__ SweepChain sweep_chain(int warp, int nb) {
  const int mid = nb / 2;
  switch (warp) {
    case 0: return SweepChain{1, 1, 1, 0, 1, mid, false};                               // y_k -= L_k y_{k-1}, k = 1..mid
    case 1: return SweepChain{nb - 1, -1, nb - 2, nb - 1, -1, nb - 2 - mid, false};     // y_k -= U_k y_{k+1}, k = nb-2..mid+1
    case 2: return SweepChain{mid, -1, mid - 1, mid, -1, mid, true};                    // x_k -= L_{k+1}' x_{k+1}, k = mid-1..0
    default: return SweepChain{mid + 1, 1, mid + 1, mid, 1, nb - 1 - mid, true};        // x_k -= U_{k-1}' x_{k-1}, k = mid+1..nb-1
  }
}

// this lane's 8 doubles of the block in `slot`, from the slab
template <int BS, bool kColumn>
__device__ __forceinline__ void slab_block_part(const double* Lsub, int slot, int lane, double (&dst)[8]) {
  constexpr int ld = BS + 2, CPL = 8;
  const int row = lane >> 1, half = lane & 1;
  const double* p = Lsub + size_t(slot) * BS * ld + (kColumn ? size_t(half * CPL) * ld + row : size_t(row) * ld + half * CPL);
  if (!kColumn) {
    const double2* p2 = reinterpret_cast<const double2*>(p);
#pragma unroll
    for (int i = 0; i < CPL / 2; ++i) { const double2 v = p2[i]; dst[2 * i] = v.x; dst[2 * i + 1] = v.y; }
  } else {
#pragma unroll
    for (int i = 0; i < CPL; ++i) dst[i] = p[i * ld];
  }
}

// after a factorisation: every sweep warp copies the first kTmemBlocks blocks of its chain into its quadrant
template <int BS>
__device__ inline void tmem_publish(const Work& W, int nb, uint32_t tmem) {
  static_assert(BS == 16, "one warp per chain, two lanes per block row");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp < 4) {
    const SweepChain ch = sweep_chain(warp, nb);
    const uint32_t base = tmem + (static_cast<uint32_t>(32 * warp) << 16);
    const int ntm = ch.count < kTmemBlocks ? ch.count : kTmemBlocks;
    for (int i = 0; i < ntm; ++i) {
      double part[8];
      if (ch.column) slab_block_part<BS, true>(W.Lsub, ch.slot0 + i * ch.dslot, lane, part);
      else slab_block_part<BS, false>(W.Lsub, ch.slot0 + i * ch.dslot, lane, part);
      tmem_st16(base + 16 * i, part);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  __syncthreads();
}

// one chain: Tensor-Memory-fed stages first, then the (at most three) stages whose block rows were requested from
// the slab when the sweep started, then -- chains longer than that -- plain slab loads
template <int BS, bool kColumn>
__device__ __forceinline__ void run_chain_tmem(const Work& W, double* bx, const SweepChain& ch, uint32_t base, int lane) {
  constexpr int CPL = 8;
  const int row = lane >> 1, half = lane & 1;
  const bool writer = half == 0;
  const int ntm = ch.count < kTmemBlocks ? ch.count : kTmemBlocks;
#ifndef OCP_B200_CHAIN_PREFETCH
#define OCP_B200_CHAIN_PREFETCH 1   // 3: three slab stages requested when the sweep starts (the first Tensor-Memory version)
#endif
#if OCP_B200_CHAIN_PREFETCH == 3
  const int nreg = ch.count - ntm < 3 ? ch.count - ntm : 3;
  double Ra[CPL], Rb[CPL], Rc[CPL];
  if (nreg > 0) slab_block_part<BS, kColumn>(W.Lsub, ch.slot0 + ntm * ch.dslot, lane, Ra);
  if (nreg > 1) slab_block_part<BS, kColumn>(W.Lsub, ch.slot0 + (ntm + 1) * ch.dslot, lane, Rb);
  if (nreg > 2) slab_block_part<BS, kColumn>(W.Lsub, ch.slot0 + (ntm + 2) * ch.dslot, lane, Rc);
#else
  // one slab stage behind the Tensor-Memory ones, requested four stages before it is needed (an L2 latency): every
  // register held through the chain is paid for by the whole iteration loop (DESIGN.md 5.5)
  const int nreg = ch.count > ntm ? 1 : 0;
  const int ireq = ntm > 4 ? ntm - 4 : 0;
  double Ra[CPL];
#endif
  const int db = ch.dblk * BS;
  const double* srcp = bx + ch.src0 * BS + half * CPL;
  double* dstp = bx + ch.dst0 * BS + row;
  for (int i = 0; i < ntm; ++i) {
#if OCP_B200_CHAIN_PREFETCH != 3
    if (nreg > 0 && i == ireq) slab_block_part<BS, kColumn>(W.Lsub, ch.slot0 + ntm * ch.dslot, lane, Ra);
#endif
    double L[CPL];
    tmem_ld16(base + 16 * i, L);
    direct::sweep_stage<BS>(L, srcp, dstp, writer);
    srcp += db; dstp += db;
  }
#if OCP_B200_CHAIN_PREFETCH != 3
  if (nreg > 0 && ntm == 0) slab_block_part<BS, kColumn>(W.Lsub, ch.slot0, lane, Ra);
#endif
  if (nreg > 0) { direct::sweep_stage<BS>(Ra, srcp, dstp, writer); srcp += db; dstp += db; }
#if OCP_B200_CHAIN_PREFETCH == 3
  if (nreg > 1) { direct::sweep_stage<BS>(Rb, srcp, dstp, writer); srcp += db; dstp += db; }
  if (nreg > 2) { direct::sweep_stage<BS>(Rc, srcp, dstp, writer); srcp += db; dstp += db; }
#endif
  for (int i = ntm + nreg; i < ch.count; ++i) {
    double L[CPL];
    slab_block_part<BS, kColumn>(W.Lsub, ch.slot0 + i * ch.dslot, lane, L);
    direct::sweep_stage<BS>(L, srcp, dstp, writer);
    srcp += db; dstp += db;
  }
}

// K x = b in place (b = [p | block 0 | ... | block nb-1]): direct::tri_solve_twisted with the sweeps fed from Tensor Memory
template <int BS>
__device__ inline void tri_solve_twisted_tmem(const PatternDev& P, const Work& W, uint32_t tmem) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.tri_np, nb = P.tri_nb, N = nb * BS;
  constexpr int ld = BS + 2;
  const int mid = nb / 2;
  double* bx = W.b + np;
  OCP_B200_FINE_CLOCK(clk, W.phase);
  const uint32_t base = tmem + (static_cast<uint32_t>(32 * (warp & 3)) << 16);
  // (No prefetch of D_k^-1 rows by the warps that idle during the forward sweep, as direct::tri_solve_twisted does:
  // here warps 0 and 1 run the sweep and load their rows in the diagonal phase anyway, so the pass is not shorter,
  // and the 32 registers held across the sweep and the border phase cost 256 bytes of spills that the whole
  // iteration loop paid for -- 7.75 -> 7.30 ms per launch without it, profiles/README.md.)
  // forward: both chains at once (warps 0 and 1), then the second contribution to block mid
  // (the block row of the joining slot is requested AFTER warp 0's chain: requested before it, its eight doubles sit
  // in registers through the whole chain -- 7.29 -> 7.08 ms per launch for the later load, profiles/README.md)
  double Lj[8];
  if (warp < 2) run_chain_tmem<BS, false>(W, bx, sweep_chain(warp, nb), base, lane);
  if (warp == 0 && mid + 1 < nb) slab_block_part<BS, false>(W.Lsub, mid + 1, lane, Lj);
  __syncthreads();
  if (warp == 0 && mid + 1 < nb) direct::sweep_stage<BS>(Lj, bx + (mid + 1) * BS + (lane & 1) * 8, bx + mid * BS + (lane >> 1), (lane & 1) == 0);
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_FWD);
  // border: y_p = b_p - sum_k L_pk y_k, x_p = D_p^-1 y_p   (as in direct::tri_solve_twisted)
  if (np > 0) {
    const int nw = T >> 5;
    if (direct::border_rows_by_warp(np, N, nw)) {
      // whole warps per border row (3 or 2 rows each), every slab load of a warp issued before its first FMA:
      // one L2 round trip for the phase instead of one per 128-column chunk and row pass
      direct::border_rows_dispatch(W.Lp, bx, W.b, W.xp, N, warp, lane, nw);
    } else {
    const int hw = tid >> 4, hl = tid & 15, nhw = T >> 4;
    for (int r0 = 0; r0 < np; r0 += nhw) {
      const int r = r0 + hw;
      const bool have = r < np;
      const double* rowp = W.Lp + size_t(have ? r : 0) * N;
      double s0 = 0.0, s1 = 0.0;
      for (int j0 = hl; j0 < N; j0 += 128) {
        double lv[8], yv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int j = j0 + 16 * u;
          const bool ok = have && j < N;
          lv[u] = ok ? rowp[j] : 0.0;
          yv[u] = ok ? bx[j] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; u += 2) { s0 = fma(lv[u], yv[u], s0); s1 = fma(lv[u + 1], yv[u + 1], s1); }
      }
      double s = s0 + s1;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (have && hl == 0) W.xp[r] = W.b[r] - s;
    }
    }
    __syncthreads();
    direct::border_apply_inverse(W.Dp, W.xp, W.b, np, tid);
    __syncthreads();
  }
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BORDER);
  // diagonal: c_k = D_k^-1 y_k - L_pk' x_p   (in place: value computed, barrier, stored)
  {
    // up to kPass passes of T rows are computed before the one barrier that protects the in-place store, so the slab
    // loads of a later pass are in flight while the earlier pass multiplies
#ifndef OCP_B200_DIAG_PASSES
#define OCP_B200_DIAG_PASSES 1
#endif
    constexpr int kPass = OCP_B200_DIAG_PASSES;
    const int Tb = (T / BS) * BS;
    const int k1 = tid / BS, r1 = tid % BS, kstep = T / BS;
    for (int base0 = 0, k0 = k1; base0 < N; base0 += kPass * Tb, k0 += kPass * kstep) {
      double vq[kPass];
#pragma unroll
      for (int q = 0; q < kPass; ++q) {
        const int base_j = base0 + q * Tb, k = k0 + q * kstep;
        const int j = tid < Tb ? base_j + tid : N;
        double v = 0.0;
        if (j < N) {
          {
            // D_k^-1 is stored column-major (tri_factor_twisted<.., kInvT>): the row of thread (k, r1) is a stride-BS
            // gather, and the 16 threads of a block read 128 contiguous bytes per element
            const double* dk = W.Dinv + size_t(k) * BS * ld + r1;
            const double* yk = bx + k * BS;
            double dr[BS];
#pragma unroll
            for (int t = 0; t < BS; ++t) dr[t] = dk[t * BS];
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
            for (int t = 0; t < BS; t += 4) {
              s0 = fma(dr[t], yk[t], s0); s1 = fma(dr[t + 1], yk[t + 1], s1);
              s2 = fma(dr[t + 2], yk[t + 2], s2); s3 = fma(dr[t + 3], yk[t + 3], s3);
            }
            v = (s0 + s1) + (s2 + s3);
          }
          double v1 = 0.0;
          if (np == 12) {   // the border size of a 12-state reference: all loads issued before the first FMA
            double lv[12];
#pragma unroll
            for (int p = 0; p < 12; ++p) lv[p] = W.Lp[size_t(p) * N + j];
#pragma unroll
            for (int p = 0; p < 12; p += 2) { v = fma(-lv[p], W.b[p], v); v1 = fma(-lv[p + 1], W.b[p + 1], v1); }
          } else {
            int p = 0;
            for (; p + 1 < np; p += 2) {
              v = fma(-W.Lp[size_t(p) * N + j], W.b[p], v);
              v1 = fma(-W.Lp[size_t(p + 1) * N + j], W.b[p + 1], v1);
            }
            if (p < np) v = fma(-W.Lp[size_t(p) * N + j], W.b[p], v);
          }
          v += v1;
        }
        vq[q] = v;
      }
      __syncthreads();
#pragma unroll
      for (int q = 0; q < kPass; ++q) {
        const int j = tid < Tb ? base0 + q * Tb + tid : N;
        if (j < N) bx[j] = vq[q];
      }
    }
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_DIAG);
  // backward, from block mid outwards: warps 2 and 3 (their quadrants hold the column layout)
  if (warp == 2 || warp == 3) run_chain_tmem<BS, true>(W, bx, sweep_chain(warp, nb), base, lane);
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BWD);
}

template <int BS>
__device__ inline void solve_instance(const PatternDev& P, const CompactIdx& C, const ocp_b200_settings& S, const SolveArgs& A,
                                      Work& W, const Ctx& X, Reducer& R, int inst, QpResult& out, uint32_t tmem) {
  const int tid = threadIdx.x, T = blockDim.x;
  const int n = P.n, m = P.m;
  const double sigma = S.sigma, relax = S.relax;
  const uint32_t* const ar = X.ar;
  PhaseClock clk(A.phase);
  W.phase = A.phase;

  // ---- load (osqp_setup copies its inputs): values, q, bounds clamped to +-1e30 ------------
  {
    const double* hv = A.h_vals + size_t(inst) * A.ld_h;
    const double* av = A.a_vals + size_t(inst) * A.ld_a;
    const double* qv = A.q + size_t(inst) * A.ld_n;
    const double* lv = A.l + size_t(inst) * A.ld_m;
    const double* uv = A.u + size_t(inst) * A.ld_m;
    // the inputs are read once: streaming loads (evict-first), they must not displace the slabs in L2
    for (int k = tid; k < P.nnz_a; k += T) W.Aval[k] = __ldcs(av + k);
    for (int k = tid; k < P.nnz_p; k += T) { const int s = P.p_src[k]; X.psm[k] = s >= 0 ? __ldcs(hv + s) : 0.0; }
    for (int j = tid; j < n; j += T) { W.q[j] = __ldcs(qv + j); W.D[j] = 1.0; }
    double bad[1] = {0.0};
    for (int i = tid; i < m; i += T) {
      const double lo = __ldcs(lv + i), hi = __ldcs(uv + i);
      if (lo > hi) bad[0] = 1.0;
      W.l[i] = fmax(lo, -kInfty);
      W.u[i] = fmin(hi, kInfty);
      W.E[i] = 1.0;
    }
    block_reduce<1, true>(bad, R);
    if (bad[0] > 0.0) {  // osqp_setup rejects l > u; the reference then adds no usable step
      for (int j = tid; j < n; j += T) W.x[j] = 0.0;
      for (int i = tid; i < m; i += T) W.y[i] = 0.0;
      __syncthreads();
      out = QpResult{OCP_B200_QP_UNSOLVED, 0, 0, 0, 0, 0.0, 0.0, S.rho};
      return;
    }
  }
  clk.lap(OCP_B200_PHASE_LOAD);

  // ---- Ruiz equilibration (scale_data).  Shared: column scales (b), row scales (x|w), P values (z|y),
  // A values.  Slab, element j / i always touched by the same thread: q, D, E, the inf-norms of the
  // scaled A / P columns (by-products of pass k that give the column norms of pass k + 1).
  double c = 1.0;
  {
    const uint32_t* ta = ar + C.acol.tent_off;
    const uint32_t* tr2 = ar + C.arow.tent2_off;
    const uint32_t* tp = ar + C.pcol.tent_off;
    double* const cs = W.b;
    double* const rs = X.rscale;
    double* const Ps = X.psm;
    for (int pass = 0; pass < S.scaling_iters; ++pass) {
      for (int j = tid; j < n; j += T) {
        double dn = 0.0;
        if (pass == 0) {
          const PSpan sp = pspan_dev(C.pcol, ar, j);
#pragma unroll 4
          for (int kt = sp.kt0; kt < sp.kt1; ++kt) dn = fmax(dn, fabs(Ps[kt + sp.kshift]));
          const PSpan sa = pspan_dev(C.acol, ar, j);
#pragma unroll 4
          for (int kt = sa.kt0; kt < sa.kt1; ++kt) dn = fmax(dn, fabs(W.Aval[kt + sa.kshift]));
        } else {
          dn = fmax(X.cn[j], X.an[j]);
        }
        cs[j] = 1.0 / sqrt(limit_scaling(dn));
      }
      for (int i = tid; i < m; i += T) {
        const PSpan s = pspan_dev(C.arow, ar, i);
        double en = 0.0;
        if (s.qd2 >= 0) {
          const double* av = W.Aval + s.qd2;
#pragma unroll 4
          for (int kt = s.kt0; kt < s.kt1; ++kt) en = fmax(en, fabs(av[plow(tr2, kt)]));
        } else {
#pragma unroll 4
          for (int kt = s.kt0; kt < s.kt1; ++kt) en = fmax(en, fabs(W.Aval[pvalue(tr2[kt], s.q)]));
        }
        rs[i] = 1.0 / sqrt(limit_scaling(en));
      }
      __syncthreads();
      double red[2] = {0.0, 0.0};  // sum of P column norms, max |q|
      for (int j = tid; j < n; j += T) {
        const double dj = cs[j];
        const double q0 = W.q[j], d0 = W.D[j];   // slab loads issued before the column loops
        double cn = 0.0, an = 0.0;
        const PSpan sp = pspan_dev(C.pcol, ar, j);
        for (int kt = sp.kt0; kt < sp.kt1; ++kt) {
          const double v = Ps[kt + sp.kshift] * cs[pvalue(tp[kt], sp.q)] * dj;
          Ps[kt + sp.kshift] = v;
          cn = fmax(cn, fabs(v));
        }
        const PSpan sa = pspan_dev(C.acol, ar, j);
#pragma unroll 4
        for (int kt = sa.kt0; kt < sa.kt1; ++kt) {
          const double v = W.Aval[kt + sa.kshift] * (rs[pvalue(ta[kt], sa.q)] * dj);
          W.Aval[kt + sa.kshift] = v;
          an = fmax(an, fabs(v));
        }
        X.an[j] = an;      // inf-norm of the scaled A column
        X.cn[j] = cn;      // inf-norm of the scaled P column, before the cost factor
        const double qj = q0 * dj;
        W.q[j] = qj;
        W.D[j] = d0 * dj;
        red[0] += cn;
        red[1] = fmax(red[1], fabs(qj));
      }
      for (int i = tid; i < m; i += T) W.E[i] *= rs[i];
      double sum[1] = {red[0]}, mx[1] = {red[1]};
      block_reduce<1, false>(sum, R);
      block_reduce<1, true>(mx, R);
      const double ct = 1.0 / limit_scaling(fmax(sum[0] / double(n), limit_scaling(mx[0])));
      for (int k = tid; k < P.nnz_p; k += T) Ps[k] *= ct;
      for (int j = tid; j < n; j += T) { W.q[j] *= ct; X.cn[j] *= ct; }
      c *= ct;
      __syncthreads();
    }
  }
  const double cinv = 1.0 / c;

  // ---- scaled bounds, constraint types (set_rho_vec); the scaled P values move to the slab ----
  double rho = fmin(fmax(S.rho, kRhoMin), kRhoMax);
  for (int i = tid; i < m; i += T) {
    const double e = W.E[i];
    const double lo = W.l[i] * e, hi = W.u[i] * e;
    W.l[i] = lo; W.u[i] = hi;
    W.ctype[i] = constraint_type(lo, hi);
  }
  for (int k = tid; k < P.nnz_p; k += T) X.pslab[k] = X.psm[k];
  __syncthreads();
  W.Pval = X.pslab;
  Rho rv(rho);
  clk.lap(OCP_B200_PHASE_SCALE);
  direct::tri_assemble_program(P, W, rv, sigma);
  clk.lap(OCP_B200_PHASE_KKT_ASSEMBLE);
  direct::tri_factor_twisted<BS, true, true, BS == 16>(P, W);   // scratch: the iteration vectors (nothing lives there yet)
  if constexpr (BS == 16) tmem_publish<BS>(W, P.tri_nb, tmem);
  clk.lap(OCP_B200_PHASE_FACTOR);
  // ---- cold start ----
  for (int j = tid; j < n; j += T) W.x[j] = 0.0;
  for (int i = tid; i < m; i += T) { W.z[i] = 0.0; W.y[i] = 0.0; W.w[i] = 0.0; }
  __syncthreads();

  const CompactOps I{C, ar, m};
  const int interval = rho_interval(S);
  int status = OCP_B200_QP_UNSOLVED, iter = 0, solves = 0, rho_updates = 0, checks = 0, n_trace = 0;
  double prim_res = 0.0, dual_res = 0.0;
  bool done = false;

  for (iter = 1; iter <= S.admm_max_iter && !done; ++iter) {
    // ---- right-hand side of the reduced KKT system: sigma x - q + A'(rho z - y) --------------
    for (int j = tid; j < n; j += T) {
      const double qj = W.q[j];   // slab
      W.b[j] = (sigma * W.x[j] - qj) + col_dot_A(C, ar, W.Aval, W.w, j);
    }
    __syncthreads();
    clk.lap(OCP_B200_PHASE_RHS);
    if constexpr (BS == 16) tri_solve_twisted_tmem<BS>(P, W, tmem);   // b <- x~
    else direct::tri_solve_twisted<BS>(P, W);
    ++solves;
    clk.lap(OCP_B200_PHASE_SOLVE);

    // ---- x, z, y updates with relaxation and projection (update_x / update_z / update_y) ----
    const IterFlags F(S, interval, iter);
    const bool want_info = F.want_info();
    {
      const uint32_t* tc = ar + C.arow.tent_off;
      const uint32_t* tp = ar + C.arow.tent2_off;
      for (int i = tid; i < m; i += T) {
        const double lo = W.l[i], hi = W.u[i];   // slab: requested before the row product
        const PSpan s = pspan_dev(C.arow, ar, i);
        double zt = 0.0;
        if (s.qd >= 0 && s.qd2 >= 0) {   // uniform deltas in the row's region (periodic_index.h)
          const double* av = W.Aval + s.qd2;
          const double* bv = W.b + s.qd;
#pragma unroll 4
          for (int kt = s.kt0; kt < s.kt1; ++kt) zt += av[plow(tp, kt)] * bv[plow(tc, kt)];
        } else {
#pragma unroll 4
          for (int kt = s.kt0; kt < s.kt1; ++kt) zt += W.Aval[pvalue(tp[kt], s.q)] * W.b[pvalue(tc[kt], s.q)];
        }
        const signed char ct = W.ctype[i];
        const double rh = rv.of(ct);
        const double zr = relax * zt + (1.0 - relax) * W.z[i];
        const double zn = fmin(fmax(zr + rv.inv(ct) * W.y[i], lo), hi);
        const double dy = rh * (zr - zn);
        const double yn = W.y[i] + dy;
        W.y[i] = yn;
        W.z[i] = zn;
        W.w[i] = rh * zn - yn;
        if (want_info) W.dy[i] = dy;
      }
    }
    for (int j = tid; j < n; j += T) {
      const double xo = W.x[j];
      const double xn = relax * W.b[j] + (1.0 - relax) * xo;
      if (want_info) W.dx[j] = xn - xo;
      W.x[j] = xn;
    }
    __syncthreads();
    clk.lap(OCP_B200_PHASE_UPDATE);
    if (!want_info) continue;

    // ---- update_info, check_termination, adapt_rho (admm_common.cuh) -------------------------
    ++checks;
    const QpVec V = qp_vectors(W, n, m);
    double mx[kRedWidth];
    update_info(I, V, R, mx);
    prim_res = prim_residual(mx);
    dual_res = dual_residual(mx, cinv);
    if (F.can_check || F.last_iter) {
      const int st = check_termination(I, V, S, R, mx, c, cinv);
      if (F.can_check) record_trace(A, inst, n_trace, iter, prim_res, dual_res, rho, solves, st);
      if (st >= 0) { status = st; done = true; clk.lap(OCP_B200_PHASE_CHECK); continue; }
      if (F.last_iter) { status = approximate_status(S, mx, cinv); done = true; continue; }
    }
    if (F.rho_time && adapt_rho(S, mx, rho)) {
      ++rho_updates;
      rv = Rho(rho);
      // the factorisation works in the space of the iteration vectors: park x, z, y in the slab
      // (element i written and read back by the same thread)
      __syncthreads();
      for (int j = tid; j < n; j += T) X.sx[j] = W.x[j];
      for (int i = tid; i < m; i += T) { X.sz[i] = W.z[i]; X.sy[i] = W.y[i]; }
      __syncthreads();
      // (inlined a second time on purpose: an out-of-line copy shared with the set-up was measured slower,
      // 9.6 -> 9.8 ms per launch with P and W passed by value, 11.7 ms by reference)
      direct::tri_assemble_program(P, W, rv, sigma);
      direct::tri_factor_twisted<BS, true, true, BS == 16>(P, W);
      if constexpr (BS == 16) tmem_publish<BS>(W, P.tri_nb, tmem);
      for (int j = tid; j < n; j += T) W.x[j] = X.sx[j];
      for (int i = tid; i < m; i += T) {
        const double zi = X.sz[i], yi = X.sy[i];
        W.z[i] = zi; W.y[i] = yi;
        W.w[i] = rv.of(W.ctype[i]) * zi - yi;
      }
      __syncthreads();
    }
    clk.lap(OCP_B200_PHASE_CHECK);
  }
  if (!done) status = OCP_B200_QP_MAX_ITER_REACHED;
  if (A.trace && inst == 0 && tid == 0 && A.n_trace) *A.n_trace = n_trace;
  out = QpResult{status, done ? iter - 1 : S.admm_max_iter, solves, rho_updates, checks, prim_res, dual_res, rho};
  // store_solution (admm_common.cuh), written out here: the shared function, same arithmetic, costs the BS = 20
  // instantiation 16 + 48 bytes of spill stores / loads more (register allocation at the 128 cap, DESIGN.md 5.5)
  const bool has_sol = status != OCP_B200_QP_PRIMAL_INFEASIBLE && status != OCP_B200_QP_DUAL_INFEASIBLE;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);
  for (int j = tid; j < n; j += T) W.x[j] = has_sol ? W.D[j] * W.x[j] : nanv;
  for (int i = tid; i < m; i += T) W.y[i] = has_sol ? cinv * W.E[i] * W.y[i] : nanv;
  __syncthreads();
}

// persistent kernel: CTAs pull instances from A.counter
template <int BS, int kThreads, int kBlocksPerSm>
__global__ void __launch_bounds__(kThreads, kBlocksPerSm)
admm_compact_kernel(const PatternDev P, const CompactIdx C, const ocp_b200_settings S, const SolveArgs A, const int layout_flags) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red_buf[2 * (kThreads / 32) * kRedWidth];
  __shared__ int s_inst;
  __shared__ uint32_t s_tmem;
  static_assert(kThreads == 128, "four sweep warps; the tiled chain steps take thread groups of 64");
  if constexpr (BS == 16) {   // Tensor Memory for the sweep blocks: one warp allocates, the same warp frees it at the end
    if (threadIdx.x < 32) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                   ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(&s_tmem))), "n"(kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  const uint32_t tmem = BS == 16 ? s_tmem : 0u;
  double* sm = reinterpret_cast<double*>(smem_raw);
  double* gl = A.slab + size_t(blockIdx.x) * A.slab_doubles;
  const Layout L = make_layout(P, C.arena_words, layout_flags);
  Work W{};
  W.b = sm + L.b; W.x = sm + L.x; W.w = sm + L.w; W.z = sm + L.z; W.y = sm + L.y;
  W.Aval = sm + L.aval; W.ctype = reinterpret_cast<signed char*>(sm + L.ctype);
  W.Dp = sm + L.dp; W.xp = sm + L.xp; W.piv = sm + L.piv;
  W.Dp2 = sm + L.dp2; W.S = sm + L.s; W.Sp = sm + L.sp; W.stage = sm + L.stage; W.Fb = sm + L.fb;
  W.s_stride = L.s_stride; W.sp_stride = L.sp_stride; W.stage_stride = L.stage_stride;
  W.ring_bar = nullptr; W.ring_phase = nullptr; W.ring_slots = 0;
  W.Dinv = gl + L.dinv; W.Lsub = gl + L.lsub; W.Lp = gl + L.lp;
  W.q = (L.q_smem ? sm : gl) + L.q; W.l = (L.lu_smem ? sm : gl) + L.l; W.u = (L.lu_smem ? sm : gl) + L.u;
  W.D = gl + L.D; W.E = gl + L.E;
  W.Pval = gl + L.pval; W.dx = gl + L.dx; W.dy = gl + L.dy;
  W.idx = nullptr; W.phase = nullptr;
  uint32_t* ar = reinterpret_cast<uint32_t*>(sm + L.arena);
  for (int k = threadIdx.x; k < C.arena_words; k += kThreads) ar[k] = C.arena[k];
  if (kCanaryDoubles > 0 && threadIdx.x == 0)
    for (int gi = 0; gi < L.nguard; ++gi)
      for (int c = 0; c < kCanaryDoubles; ++c) ((L.guard_slab[gi] ? gl : sm) + L.guard_off[gi])[c] = canary_value(gi);
  Ctx X{ar, sm + L.rscale, sm + L.psm, gl + L.an, gl + L.cn, gl + L.sx, gl + L.sz, gl + L.sy, gl + L.pval};
  __syncthreads();
  Reducer R{red_buf, 0, (kThreads / 32) * kRedWidth};
  for (int inst; (inst = next_instance(A, s_inst)) < A.B;) {
    QpResult res;
    solve_instance<BS>(P, C, S, A, W, X, R, inst, res, tmem);
    write_outputs(P, A, W.x, W.y, R, inst, res);
  }
  if constexpr (BS == 16) {
    __syncthreads();
    if (threadIdx.x < 32)
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
  }
  if (kCanaryDoubles > 0 && threadIdx.x == 0)
    for (int gi = 0; gi < L.nguard; ++gi)
      for (int c = 0; c < kCanaryDoubles; ++c)
        if (__double_as_longlong(((L.guard_slab[gi] ? gl : sm) + L.guard_off[gi])[c]) != __double_as_longlong(canary_value(gi)))
          printf("OCP_B200 CANARY overwritten: compact kernel, guard %d (%s), CTA %d\n", gi, L.guard_slab[gi] ? "slab" : "shared", int(blockIdx.x));
}

}  // namespace compact
}  // namespace ocpb200
