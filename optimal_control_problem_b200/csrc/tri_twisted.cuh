// tri_twisted.cuh -- "burn at both ends" (twisted) variant of the bordered block-tridiagonal
// LDL' of admm_direct_kernel.cuh, exact block size BS.
//
// The factorisation and the two sweeps of a solve are sequential in the block index, and one
// warp cannot go faster than its dependent-instruction chain.  The twisted ordering eliminates
// blocks 0, 1, ..., mid-1 from the top and nb-1, nb-2, ..., mid+1 from the bottom AT THE SAME
// TIME (two thread groups / two warps), and block mid last.  Same storage, no extra fill, half
// the sequential depth:
//     top    k = 1..mid      L_k = K_{k,k-1} D_{k-1}^-1      D_k -= L_k K_{k,k-1}'
//     bottom k = nb-2..mid   U_k = K_{k,k+1} D_{k+1}^-1      D_k -= U_k K_{k+1,k}
// Slot s of the sub-diagonal storage (which starts out as K_{s,s-1}) ends up holding L_s for
// s <= mid and U_{s-1} for s > mid.  The border rows (reference parameters) follow either
// chain with the same recurrences:  V_k -= V_pred C',  L_p,pred = V_pred D_pred^-1,
// D_p -= V_pred L_p,pred', where C is the coupling block just computed.
#pragma once

namespace ocpb200 {
namespace direct {

__device__ __forceinline__ void group_barrier(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// One elimination step of a chain, executed by a thread group (gt of GT threads, barrier `bar`):
//   C  = slot content: K_{s,s-1}; the step owns block k, the previously eliminated neighbour is `pred`
//   kTop: k = s, pred = s - 1, coupling = C Dinv_pred;  else: k = s - 1, pred = s, coupling = C' Dinv_pred
// Updates D_k (not inverted here), V_k, finalises L_p,pred, accumulates into Dpacc, overwrites the slot.
// kStaged: the caller guarantees stage != nullptr and F != nullptr (the compact kernel): without the run-time choice
// between a global and a shared-memory operand the compiler keeps the address space of both and the dot products
// load with LDS instead of generic loads.
// kTile: the dot products as 2 x 2 tiles (tri_fast.cuh: same bits, a third of the shared-memory loads) -- for thread
// groups of at most BS * BS / 4 threads, where every thread has at least four results per loop anyway.
// kInvT: the inverted blocks D_pred^-1 are stored column-major with pitch BS (warp_invert_exact<.., true>); the staging
// copy transposes D_pred^-1 back to the row layout the dot products read.
template <int BS, bool kTop, bool kStaged = false, bool kTile = false, bool kInvT = false>
__device__ __forceinline__ void chain_step(const Work& W, int np, int N, int /*ld*/, int k, int pred, int slot, double* S,
                                           double* Sp, double* Dpacc, int gt, int GT, int bar, double* stage, double* F = nullptr) {
  constexpr int bb = BS * BS, ld = BS + 2;   // compile-time pitch: addresses fold into immediates
  const int pb = np * BS;
  double* Cg = W.Lsub + size_t(slot) * BS * ld;
  double* Dk = W.Dinv + size_t(k) * BS * ld;
  const double* Dg = W.Dinv + size_t(pred) * BS * ld;   // D_pred^-1 (symmetric)
  // With the factor in the global slab every dot product below would re-read block rows from L2:
  // copy the two blocks this step multiplies into shared memory once (coalesced 16-byte loads).
  const double* C = Cg;
  const double* Dm = Dg;
  static_assert(!kInvT || kStaged, "a column-major D^-1 is read through the staging copy");
  if (kStaged || stage != nullptr) {
    double2* cs = reinterpret_cast<double2*>(stage);
    double2* ds = reinterpret_cast<double2*>(stage + W.stage_stride);
    const double2* cg2 = reinterpret_cast<const double2*>(Cg);
    const double2* dg2 = reinterpret_cast<const double2*>(Dg);
    if constexpr (kInvT) {
      for (int e = gt; e < BS * ld / 2; e += GT) cs[e] = cg2[e];
      double* dd = stage + W.stage_stride;
      for (int e = gt; e < bb; e += GT) dd[(e % BS) * ld + e / BS] = Dg[e];
    } else {
      for (int e = gt; e < BS * ld / 2; e += GT) { cs[e] = cg2[e]; ds[e] = dg2[e]; }
    }
    group_barrier(bar, GT);
    C = stage; Dm = stage + W.stage_stride;
  }
  // coupling block into S; V_pred into Sp
  if constexpr (kTile) {
    for (int e = gt; e < bb / 4; e += GT) {
      const int r0 = 2 * (e / (BS / 2)), c0 = 2 * (e % (BS / 2));
      double o[4];
      if (kTop) {
        tile_cc<BS>(C + r0 * ld, C + (r0 + 1) * ld, Dm + c0 * ld, Dm + (c0 + 1) * ld, o);
        S[r0 * ld + c0] = o[0]; S[r0 * ld + c0 + 1] = o[1]; S[(r0 + 1) * ld + c0] = o[2]; S[(r0 + 1) * ld + c0 + 1] = o[3];
      } else {   // o[2 i + j] = sum_t Dm[c0 + i][t] C[t][r0 + j] = S[r0 + j][c0 + i]
        tile_cs<BS>(Dm + c0 * ld, Dm + (c0 + 1) * ld, C + r0, ld, o);
        S[r0 * ld + c0] = o[0]; S[(r0 + 1) * ld + c0] = o[1]; S[r0 * ld + c0 + 1] = o[2]; S[(r0 + 1) * ld + c0 + 1] = o[3];
      }
    }
  } else {
  for (int e = gt; e < bb; e += GT) {
    const int r = e / BS, c = e % BS;
    S[r * ld + c] = kTop ? dot_cc<BS>(C + r * ld, Dm + c * ld) : dot_cs<BS>(Dm + c * ld, C + r, ld);
  }
  }
  for (int e = gt; e < pb; e += GT) {
    const int r = e / BS, c = e % BS;
    Sp[e] = W.Lp[size_t(r) * N + pred * BS + c];
  }
  group_barrier(bar, GT);
  // D_k -= coupling * K_{pred,k};  V_k -= V_pred coupling';  L_p,pred = V_pred D_pred^-1
  const bool tile_p = kTile && (np & 1) == 0;   // border loops in tiles: even border size
  if constexpr (kTile) {
    for (int e = gt; e < bb / 4; e += GT) {
      const int r0 = 2 * (e / (BS / 2)), c0 = 2 * (e % (BS / 2));
      double o[4];
      if (kTop) tile_cc<BS>(S + r0 * ld, S + (r0 + 1) * ld, C + c0 * ld, C + (c0 + 1) * ld, o);
      else tile_cs<BS>(S + r0 * ld, S + (r0 + 1) * ld, C + c0, ld, o);
      Dk[r0 * ld + c0] -= o[0]; Dk[r0 * ld + c0 + 1] -= o[1]; Dk[(r0 + 1) * ld + c0] -= o[2]; Dk[(r0 + 1) * ld + c0 + 1] -= o[3];
    }
  } else {
  for (int e = gt; e < bb; e += GT) {
    const int r = e / BS, c = e % BS;
    Dk[r * ld + c] -= kTop ? dot_cc<BS>(S + r * ld, C + c * ld) : dot_cs<BS>(S + r * ld, C + c, ld);
  }
  }
  if (tile_p) {
    for (int e = gt; e < pb / 4; e += GT) {
      const int r0 = 2 * (e / (BS / 2)), c0 = 2 * (e % (BS / 2));
      double so[4], fo[4];
      tile_cc<BS>(Sp + r0 * BS, Sp + (r0 + 1) * BS, S + c0 * ld, S + (c0 + 1) * ld, so);
      tile_cc<BS>(Sp + r0 * BS, Sp + (r0 + 1) * BS, Dm + c0 * ld, Dm + (c0 + 1) * ld, fo);
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int r = r0 + i, c = c0 + j;
          W.Lp[size_t(r) * N + k * BS + c] -= so[2 * i + j];
          W.Lp[size_t(r) * N + pred * BS + c] = fo[2 * i + j];
          if (kStaged || F != nullptr) F[r * BS + c] = fo[2 * i + j];
        }
    }
  } else {
  for (int e = gt; e < pb; e += GT) {
    const int r = e / BS, c = e % BS;
    const double s = dot_cc<BS>(Sp + r * BS, S + c * ld);
    const double f = dot_cc<BS>(Sp + r * BS, Dm + c * ld);
    W.Lp[size_t(r) * N + k * BS + c] -= s;
    W.Lp[size_t(r) * N + pred * BS + c] = f;
    if (kStaged || F != nullptr) F[e] = f;   // shared-memory copy of L_p,pred for the accumulation below (L_p may live in the slab)
  }
  }
  group_barrier(bar, GT);
  // D_p accumulator += V_pred L_p,pred';  slot <- coupling
  if (tile_p && (kStaged || F != nullptr)) {
    const int hp = np / 2;
    for (int e = gt; e < hp * hp; e += GT) {
      const int r0 = 2 * (e / hp), c0 = 2 * (e - (e / hp) * hp);
      double o[4];
      tile_cc<BS>(Sp + r0 * BS, Sp + (r0 + 1) * BS, F + c0 * BS, F + (c0 + 1) * BS, o);
      Dpacc[r0 * (np + 1) + c0] += o[0]; Dpacc[r0 * (np + 1) + c0 + 1] += o[1];
      Dpacc[(r0 + 1) * (np + 1) + c0] += o[2]; Dpacc[(r0 + 1) * (np + 1) + c0 + 1] += o[3];
    }
  } else {
  for (int e = gt; e < np * np; e += GT) {
    const int r = e / np, c = e - r * np;
    Dpacc[r * (np + 1) + c] += (kStaged || F != nullptr) ? dot_cc<BS>(Sp + r * BS, F + c * BS)
                                            : dot_cs<BS>(Sp + r * BS, W.Lp + size_t(c) * N + pred * BS, 1);
  }
  }
  for (int e = gt; e < bb; e += GT) {
    const int r = e / BS, c = e % BS;
    Cg[r * ld + c] = S[r * ld + c];
  }
  group_barrier(bar, GT);
}

template <int BS, bool kStaged = false, bool kTile = false, bool kInvT = false>
__device__ inline void tri_factor_twisted(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31;
  const int np = P.tri_np, nb = P.tri_nb, N = nb * BS;
  constexpr int ld = BS + 2;   // == P.tri_ld for even BS (checked by the dispatcher)
  const int mid = nb / 2;
  const int GT = T / 2;                    // two thread groups of whole warps
  const int grp = tid >= GT ? 1 : 0, gt = tid - grp * GT;
  double* S = W.S + grp * W.s_stride;
  double* Sp = W.Sp + grp * W.sp_stride;
  double* piv = W.piv + grp * 32;
  double* Dpacc = W.Dp2 + grp * np * (np + 1);
  double* stage = (kStaged || W.stage) ? W.stage + grp * 2 * W.stage_stride : nullptr;
  double* F = (kStaged || W.Fb) ? W.Fb + grp * W.sp_stride : nullptr;   // shared-memory copy of the L_p block just finished (optional)
  for (int e = gt; e < np * (np + 1); e += GT) Dpacc[e] = 0.0;
  // both chains: invert the chain's current block, then eliminate into the next one
  if (grp == 0) {
    OCP_B200_FINE_CLOCK(clk, W.phase);
    for (int k = 0; k < mid; ++k) {           // blocks 0..mid-1; step into k+1 (the last one is mid)
      if (gt < 32) warp_invert_exact<BS, BS + 2, kInvT>(W.Dinv + size_t(k) * BS * ld, ld, lane, piv);
      group_barrier(1, GT);
      OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_FACTOR_INVERT);
      chain_step<BS, true, kStaged, kTile, kInvT>(W, np, N, ld, k + 1, k, k + 1, S, Sp, Dpacc, gt, GT, 1, stage, F);
      OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_FACTOR_STEP);
    }
  } else {
    for (int k = nb - 1; k > mid + 1; --k) {  // blocks nb-1..mid+2; step into k-1 (>= mid+1)
      if (gt < 32) warp_invert_exact<BS, BS + 2, kInvT>(W.Dinv + size_t(k) * BS * ld, ld, lane, piv);
      group_barrier(2, GT);
      chain_step<BS, false, kStaged, kTile, kInvT>(W, np, N, ld, k - 1, k, k, S, Sp, Dpacc, gt, GT, 2, stage, F);
    }
    if (mid + 1 < nb) {                       // block mid+1: inverted here, eliminated into mid below
      if (gt < 32) warp_invert_exact<BS, BS + 2, kInvT>(W.Dinv + size_t(mid + 1) * BS * ld, ld, lane, piv);
      group_barrier(2, GT);
    }
  }
  __syncthreads();
  // the bottom chain's last step lands on block mid as well: run it with the whole CTA
  if (mid + 1 < nb) chain_step<BS, false, kStaged, kTile, kInvT>(W, np, N, ld, mid, mid + 1, mid + 1, W.S, W.Sp, W.Dp2, tid, T, 0, W.stage, W.Fb);
  if (tid < 32) warp_invert_exact<BS, BS + 2, kInvT>(W.Dinv + size_t(mid) * BS * ld, ld, lane, W.piv);
  __syncthreads();
  // border of the last block, then D_p = K_pp - (accumulated) - V_mid L_p,mid', inverted
  if (np > 0) {
    const double* Dm = W.Dinv + size_t(mid) * BS * ld;
    const int pb = np * BS;
    for (int e = tid; e < pb; e += T) {
      const int r = e / BS, c = e % BS;
      W.Sp[e] = W.Lp[size_t(r) * N + mid * BS + c];
    }
    __syncthreads();
    for (int e = tid; e < pb; e += T) {
      const int r = e / BS, c = e % BS;
      const double f = kInvT ? dot_cs<BS>(W.Sp + r * BS, Dm + c, BS) : dot_cc<BS>(W.Sp + r * BS, Dm + c * ld);
      W.Lp[size_t(r) * N + mid * BS + c] = f;
      if (kStaged || W.Fb != nullptr) W.Fb[e] = f;
    }
    __syncthreads();
    for (int e = tid; e < np * np; e += T) {
      const int r = e / np, c = e - r * np;
      const int o = r * (np + 1) + c;
      W.Dp[o] -= W.Dp2[o] + W.Dp2[np * (np + 1) + o] +
                 ((kStaged || W.Fb != nullptr) ? dot_cc<BS>(W.Sp + r * BS, W.Fb + c * BS)
                                  : dot_cs<BS>(W.Sp + r * BS, W.Lp + size_t(c) * N + mid * BS, 1));
    }
    __syncthreads();
    if (tid < 32) invert_border(W.Dp, np, lane, W.piv);
    __syncthreads();
  }
}

// one sweep stage out of a ring slot, one lane per block row (CPL == BS): every shared-memory load is
// issued before the first FMA -- the stream of a single warp is in-order, a load placed behind an
// FMA that waits for its operands costs a full shared-memory latency
template <int BS, bool kColumn>
__device__ __forceinline__ void ring_stage(const double* __restrict__ blk, const double* __restrict__ src,
                                           double* __restrict__ dst, bool writer, bool src_vec) {
  constexpr int ld = BS + 2;
  static_assert(TriCfg<BS>::LPR == 1 && BS % 4 == 0, "one lane per row");
  double lv[BS], sv[BS];
  if (!kColumn) {
    const double2* p2 = reinterpret_cast<const double2*>(blk);
#pragma unroll
    for (int i = 0; i < BS / 2; ++i) { const double2 v = p2[i]; lv[2 * i] = v.x; lv[2 * i + 1] = v.y; }
  } else {
#pragma unroll
    for (int i = 0; i < BS; ++i) lv[i] = blk[i * ld];
  }
  if (src_vec) {
    const double2* q2 = reinterpret_cast<const double2*>(src);
#pragma unroll
    for (int i = 0; i < BS / 2; ++i) { const double2 v = q2[i]; sv[2 * i] = v.x; sv[2 * i + 1] = v.y; }
  } else {
#pragma unroll
    for (int i = 0; i < BS; ++i) sv[i] = src[i];
  }
  const double old = writer ? *dst : 0.0;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
  for (int c = 0; c < BS; c += 4) {
    s0 = fma(lv[c], sv[c], s0); s1 = fma(lv[c + 1], sv[c + 1], s1);
    s2 = fma(lv[c + 2], sv[c + 2], s2); s3 = fma(lv[c + 3], sv[c + 3], s3);
  }
  if (writer) *dst = old - ((s0 + s1) + (s2 + s3));
  __syncwarp();
}

// `count` consecutive sweep stages by one warp: stage i multiplies slot (slot0 + i*dslot) with
// source block (src0 + i*dblk) and subtracts from destination block (dst0 + i*dblk).
// kColumn = false: dst[r] -= sum_c M[r][c] src[c]   (forward sweeps)
// kColumn = true : dst[r] -= sum_c M[c][r] src[c]   (backward sweeps)
template <int BS, bool kColumn>
__device__ __forceinline__ void run_chain(const Work& W, double* bx, int /*ld*/, int slot0, int dslot, int dst0, int src0,
                                          int dblk, int count, int lane, int chain) {
  constexpr int CPL = TriCfg<BS>::CPL, LPR = TriCfg<BS>::LPR, ld = BS + 2;
  const int row = lane / LPR, half = lane % LPR;
  const bool act = row < BS;
  const int rr = act ? row : 0;
  const bool writer = act && half == 0;
  if (count <= 0) return;
  // everything advances by pointer increments: no per-stage multiplications in the single warp's stream
  const double* lp = W.Lsub + size_t(slot0) * BS * ld + (kColumn ? size_t(half * CPL) * ld + rr : size_t(rr) * ld + half * CPL);
  const int dl = dslot * BS * ld, db = dblk * BS;
  const double* srcp = bx + src0 * BS + half * CPL;
  double* dstp = bx + dst0 * BS + rr;
  auto load = [&](double (&dst)[CPL], const double* p) {
    if (!kColumn) {
      const double2* p2 = reinterpret_cast<const double2*>(p);
#pragma unroll
      for (int i = 0; i < CPL / 2; ++i) { const double2 v = p2[i]; dst[2 * i] = v.x; dst[2 * i + 1] = v.y; }
    } else {
#pragma unroll
      for (int i = 0; i < CPL; ++i) dst[i] = p[i * ld];
    }
  };
  if constexpr (CPL > 8) if (W.ring_slots >= 2) {
    // slab-resident factor, wide block rows: blocks arrive through the shared-memory ring
    const int R = W.ring_slots, stride = W.stage_stride;
    double* ring = W.stage + chain * R * stride;
    unsigned long long* bars = W.ring_bar + chain * kMaxRing;
    constexpr uint32_t bytes = BS * ld * sizeof(double);
    const double* gp = W.Lsub + size_t(slot0) * BS * ld;
    uint32_t ph = W.ring_phase[chain];
    if (lane == 0)
      for (int i = 0; i < R && i < count; ++i) ring_issue(ring + i * stride, gp + i * dl, bytes, bars + i);
    const int off = kColumn ? (half * CPL) * ld + rr : rr * ld + half * CPL;
    const bool src_vec = (reinterpret_cast<unsigned long long>(srcp) & 15ULL) == 0ULL;   // uniform: np even
    int s = 0;
    for (int i = 0; i < count; ++i) {
      ring_wait(bars + s, (ph >> s) & 1u);
      ph ^= 1u << s;
      ring_stage<BS, kColumn>(ring + s * stride + off, srcp, dstp, writer, src_vec);   // ends with __syncwarp
      if (lane == 0 && i + R < count) ring_issue(ring + s * stride, gp + (i + R) * dl, bytes, bars + s);
      srcp += db; dstp += db;
      s = s + 1 == R ? 0 : s + 1;
    }
    if (lane == 0) W.ring_phase[chain] = ph;
    __syncwarp();
    return;
  }
  if (W.stage != nullptr && CPL <= 8) {
    // slab-resident factor: three register buffers, block rows requested two stages ahead (an L2
    // round trip under load is longer than one stage)
    double La[CPL], Lb[CPL], Lc[CPL];
    load(La, lp);
    if (count > 1) load(Lb, lp + dl);
    for (int i = 0; i < count; i += 3) {
      if (i + 2 < count) load(Lc, lp + 2 * dl);
      sweep_stage<BS>(La, srcp, dstp, writer);
      if (i + 1 < count) {
        if (i + 3 < count) load(La, lp + 3 * dl);
        sweep_stage<BS>(Lb, srcp + db, dstp + db, writer);
      }
      if (i + 2 < count) {
        if (i + 4 < count) load(Lb, lp + 4 * dl);
        sweep_stage<BS>(Lc, srcp + 2 * db, dstp + 2 * db, writer);
      }
      lp += 3 * dl; srcp += 3 * db; dstp += 3 * db;
    }
    return;
  }
  double La[CPL], Lb[CPL];
  load(La, lp);
  for (int i = 0; i < count; i += 2) {
    if (i + 1 < count) load(Lb, lp + dl);
    sweep_stage<BS>(La, srcp, dstp, writer);
    if (i + 1 < count) {
      if (i + 2 < count) load(La, lp + 2 * dl);
      sweep_stage<BS>(Lb, srcp + db, dstp + db, writer);
    }
    lp += 2 * dl; srcp += 2 * db; dstp += 2 * db;
  }
}

// border rows of a solve, RW rows per warp: y_p[r] = b_p[r] - sum_j L_p[r][j] y[j] for N <= 320 columns.  The order of
// the sum of a row does not depend on RW, so every launch plan that takes this path gives the same bits.
template <int RW, bool kExact>   // kExact: N == 320, no index clamps
__device__ __forceinline__ void border_rows_warp(const double* __restrict__ Lp, const double* __restrict__ y,
                                                 const double* __restrict__ bp, double* __restrict__ xp, int N, int warp,
                                                 int lane) {
  constexpr int U = 10;
  double lv[RW][U];
#pragma unroll
  for (int r = 0; r < RW; ++r) {
    const double* rowp = Lp + size_t(warp * RW + r) * N;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      // (clamped index + select: a conditional load costs a branch region per element)
      const int j = lane + 32 * u;
      const double v = rowp[kExact || j < N ? j : N - 1];
      lv[r][u] = kExact || j < N ? v : 0.0;
    }
  }
  double yv[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int j = lane + 32 * u;
    const double v = y[kExact || j < N ? j : N - 1];
    yv[u] = kExact || j < N ? v : 0.0;
  }
  double s[RW];
#pragma unroll
  for (int r = 0; r < RW; ++r) {
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int u = 0; u < U; u += 2) { s0 = fma(lv[r][u], yv[u], s0); s1 = fma(lv[r][u + 1], yv[u + 1], s1); }
    s[r] = s0 + s1;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int r = 0; r < RW; ++r) s[r] += __shfl_xor_sync(0xffffffffu, s[r], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < RW; ++r) xp[warp * RW + r] = bp[warp * RW + r] - s[r];
  }
}

__device__ __forceinline__ bool border_rows_by_warp(int np, int N, int nw) {
  return np == 12 && N <= 320 && (nw == 4 || nw == 6 || nw == 12);
}

template <bool kExact>
__device__ __forceinline__ void border_rows_pick(const double* Lp, const double* y, const double* bp, double* xp, int N,
                                                 int warp, int lane, int nw) {
  if (nw == 4) border_rows_warp<3, kExact>(Lp, y, bp, xp, N, warp, lane);
  else if (nw == 6) border_rows_warp<2, kExact>(Lp, y, bp, xp, N, warp, lane);
  else border_rows_warp<1, kExact>(Lp, y, bp, xp, N, warp, lane);
}
__device__ __forceinline__ void border_rows_dispatch(const double* Lp, const double* y, const double* bp, double* xp, int N,
                                                     int warp, int lane, int nw) {
  if (N == 320) border_rows_pick<true>(Lp, y, bp, xp, N, warp, lane, nw);
  else border_rows_pick<false>(Lp, y, bp, xp, N, warp, lane, nw);
}

// x_p = D_p^-1 y_p by the first np threads (after the barrier that publishes y_p in xp)
__device__ __forceinline__ void border_apply_inverse(const double* Dp, const double* xp, double* b, int np, int tid) {
  if (tid >= np) return;
  if (np == 12) {   // the border size of a 12-state reference: every load issued before the first FMA
    double d[12], x[12];
#pragma unroll
    for (int c = 0; c < 12; ++c) { d[c] = Dp[tid * 13 + c]; x[c] = xp[c]; }
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int c = 0; c < 12; c += 2) { s0 = fma(d[c], x[c], s0); s1 = fma(d[c + 1], x[c + 1], s1); }
    b[tid] = s0 + s1;
    return;
  }
  double s0 = 0.0, s1 = 0.0;
  int c = 0;
  for (; c + 1 < np; c += 2) {
    s0 = fma(Dp[tid * (np + 1) + c], xp[c], s0);
    s1 = fma(Dp[tid * (np + 1) + c + 1], xp[c + 1], s1);
  }
  if (c < np) s0 = fma(Dp[tid * (np + 1) + c], xp[c], s0);
  b[tid] = s0 + s1;
}

// K x = b in place: b is [p | block 0 | ... | block nb-1]
template <int BS>
__device__ inline void tri_solve_twisted(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  const int np = P.tri_np, nb = P.tri_nb, N = nb * BS;
  constexpr int ld = BS + 2;
  const int mid = nb / 2;
  double* bx = W.b + np;
  OCP_B200_FINE_CLOCK(clk, W.phase);
  // The diagonal phase needs one row of D_k^-1 per thread; with the factor in the global slab that
  // is an L2 round trip on the critical path.  The warps that idle during the forward sweep fetch
  // their row now (first pass of the diagonal phase only) and keep it in registers.
  const int dTb = (T / BS) * BS;
  const bool pre = W.stage != nullptr && warp >= 2 && tid < dTb && tid < N;   // slab-resident factor only
  double drow[BS];
  if (pre) {
    const double2* p2 = reinterpret_cast<const double2*>(W.Dinv + size_t(tid / BS) * BS * ld + (tid % BS) * ld);
#pragma unroll
    for (int i = 0; i < BS / 2; ++i) { const double2 v = p2[i]; drow[2 * i] = v.x; drow[2 * i + 1] = v.y; }
  }
  // forward: top chain y_k = b_k - L_k y_{k-1} (k = 1..mid-1) and bottom chain
  // y_k = b_k - U_k y_{k+1} (k = nb-2..mid+1) on two warps, then both contributions to block mid
  if (warp == 0) run_chain<BS, false>(W, bx, ld, 1, 1, 1, 0, 1, mid - 1, lane, 0);
  else if (warp == 1) run_chain<BS, false>(W, bx, ld, nb - 1, -1, nb - 2, nb - 1, -1, nb - 2 - mid, lane, 1);
  __syncthreads();
  if (warp == 0) {
    if (mid >= 1) run_chain<BS, false>(W, bx, ld, mid, 1, mid, mid - 1, 1, 1, lane, 0);
    if (mid + 1 < nb) run_chain<BS, false>(W, bx, ld, mid + 1, 1, mid, mid + 1, 1, 1, lane, 0);
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_FWD);
  // border: y_p = b_p - sum_k L_pk y_k, x_p = D_p^-1 y_p.  Twelve border rows (a 12-state reference): whole warps
  // per row, every load before the first FMA (border_rows_warp); otherwise half a warp per border row, loads
  // issued in batches of 8 so that a slab-resident L_p costs one L2 latency per batch
  if (np > 0) {
    if (border_rows_by_warp(np, N, nw)) {
      border_rows_dispatch(W.Lp, bx, W.b, W.xp, N, warp, lane, nw);
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
    border_apply_inverse(W.Dp, W.xp, W.b, np, tid);
    __syncthreads();
  }
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BORDER);
  // diagonal: c_k = D_k^-1 y_k - L_pk' x_p   (in place: value computed, barrier, stored)
  {
    const int Tb = (T / BS) * BS;   // whole blocks per pass: a pass never reads what it overwrites
    const int k1 = tid / BS, r1 = tid % BS, kstep = T / BS;
    for (int base = 0, k = k1; base < N; base += Tb, k += kstep) {
      const int j = tid < Tb ? base + tid : N;
      double v = 0.0;
      if (j < N) {
        if (pre && base == 0) {
          const double* yk = bx + k * BS;
          double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
          for (int t = 0; t < BS; t += 4) {
            s0 = fma(drow[t], yk[t], s0); s1 = fma(drow[t + 1], yk[t + 1], s1);
            s2 = fma(drow[t + 2], yk[t + 2], s2); s3 = fma(drow[t + 3], yk[t + 3], s3);
          }
          v = (s0 + s1) + (s2 + s3);
        } else {
          v = dot_cs<BS>(W.Dinv + size_t(k) * BS * ld + r1 * ld, bx + k * BS, 1);
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
      __syncthreads();
      if (j < N) bx[j] = v;
    }
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_DIAG);
  // backward, from block mid outwards: x_k = c_k - L_{k+1}' x_{k+1} (k = mid-1..0) and
  // x_k = c_k - U_{k-1}' x_{k-1} (k = mid+1..nb-1)
  if (warp == 0) run_chain<BS, true>(W, bx, ld, mid, -1, mid - 1, mid, -1, mid, lane, 0);
  else if (warp == 1) run_chain<BS, true>(W, bx, ld, mid + 1, 1, mid + 1, mid, 1, nb - 1 - mid, lane, 1);
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BWD);
}

}  // namespace direct
}  // namespace ocpb200
