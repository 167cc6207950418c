// admm_direct_kernel.cuh -- batched ADMM QP solver for sm_100a with a DIRECT reduced-KKT solve.
//
// Replaces, for B independent QPs that share one sparsity pattern, what the reference does per
// SQP step through OsqpEigen/OSQP (src/sqp_solver/CuCaQP.cpp:271-288, 183-224): osqp_setup
// (bound clamping, Ruiz equilibration x10 with cost normalisation, rho vector, factorisation,
// cold start) and osqp_solve (ADMM iterations, residual / termination / infeasibility checks
// every 25 iterations, adaptive rho, unscaling), then the SQP update x += alpha * d[np:]
// (SQPOptimizationSolver.cpp:171-177).
//
// Linear system.  OSQP's reduced ("indirect") KKT matrix
//     K = P + sigma I + A' diag(rho) A
// of a multiple-shooting OCP is block tridiagonal in the stage index (dynamics rows couple
// stage k with k+1 only) with a dense border for the reference parameters p, which every
// stage cost may touch.  With the p columns ordered last, K = L D L' with dense bs x bs
// blocks has no fill outside that structure:
//     D_k   = K_kk - L_k D_{k-1} L_k'            L_k   = K_{k,k-1} D_{k-1}^-1
//     V_k   = K_pk - V_{k-1} L_k'                L_pk  = V_k D_k^-1
//     D_p   = K_pp - sum_k V_k L_pk'
// The kernel keeps D_k^-1 (explicit, Gauss-Jordan), L_k and L_pk, so that a solve is two
// sequential sweeps of dense bs x bs mat-vecs (one warp) plus fully parallel dense work.  The
// solve is exact up to rounding, like the LDL' of the full KKT system that the reference's CPU
// build of OSQP uses (oracle/osqp_restate.hpp) -- the ADMM iterates of the two agree to
// rounding, which is what the parity tests check.
//
// Layout.  One persistent CTA per SM takes instances from an atomic counter.  Per-instance
// state is a list of arrays (vectors, matrix values, factor blocks, index structures); a
// host-side plan puts as many of them as fit into shared memory, in priority order, and the
// rest into a per-CTA slab of global memory that stays L2-resident.  For the H=20 quadrotor
// everything is in shared memory and an ADMM iteration touches no DRAM at all.  Termination,
// rho updates and refactorisations are decided on the device: one launch per SQP step.
#pragma once

#include "admm_common.cuh"
#include "block_ring.cuh"
#include "direct_layout.cuh"

namespace ocpb200 {
namespace direct {

constexpr int kMaxRing = 8;   // ring slots per chain

struct Work {
  double *x, *q, *b, *z, *y, *l, *u;
  signed char* ctype;
  double *Aval, *Dinv, *Lsub;
  idx_t* idx;
  double *Pval;
  double *stage;   // block staging buffers (null when the factor is in shared memory anyway)
  int stage_stride;
  // asynchronous block ring of the sweeps (tri_twisted.cuh): the staging buffers split between the two
  // chains, one mbarrier per slot, the phase parity of every slot kept across calls
  unsigned long long* ring_bar;
  unsigned* ring_phase;
  int ring_slots;   // per chain; 0 = no ring
  double *Lp, *Dp, *Dp2, *S, *Sp, *xp, *piv;   // border: L_pk [np x N], D_p^-1 [np x (np+1)], scratch (two sets)
  double* Fb;   // optional: two [np x bs] shared-memory tiles holding the L_p block a chain step just finished (null: read it back from L_p)
  int s_stride, sp_stride;
  long long* phase;   // cycle counters of CTA 0 (null unless profiling)
  double *w;                        // rho .* z - y, kept current by the update phase
  double *D, *E, *dx, *dy;
};

// With a compile-time placement (PLACE_SMEM / PLACE_MULTI) every pointer is derived from exactly
// one base, so the compiler knows its address space and emits LDS/STS or LDG/STG, not generic LD.
template <int kPlace>
__device__ __forceinline__ void carve(Work& W, const PatternDev& P, uint32_t smem_mask, double* sm, double* gl, bool check = false) {
  double* ptr[AR_COUNT];
#pragma unroll
  for (int id = 0; id < AR_COUNT; ++id) {
    const size_t sz = slot_doubles(P, kPlace, id);
    const bool in_smem = ((kPlace == PLACE_MIXED ? smem_mask : placement_mask(kPlace)) >> id & 1u) != 0;
    if (in_smem) { ptr[id] = sm; sm += sz; }
    else { ptr[id] = gl; gl += sz; }
    if (kCanaryDoubles > 0 && sz > 0) {   // guard doubles at the end of the array's slot
      double* g = (in_smem ? sm : gl) - kCanaryDoubles;
      if (check) {
        if (threadIdx.x == 0)
          for (int c = 0; c < kCanaryDoubles; ++c)
            if (__double_as_longlong(g[c]) != __double_as_longlong(canary_value(id)))
              printf("OCP_B200 CANARY overwritten: direct kernel placement %d, array %d, CTA %d\n", kPlace, id, int(blockIdx.x));
      } else if (threadIdx.x == 0) {
        for (int c = 0; c < kCanaryDoubles; ++c) g[c] = canary_value(id);
      }
    }
  }
  W.x = ptr[AR_X]; W.q = ptr[AR_Q]; W.b = ptr[AR_B]; W.z = ptr[AR_Z]; W.y = ptr[AR_Y]; W.l = ptr[AR_L]; W.u = ptr[AR_U];
  W.ctype = reinterpret_cast<signed char*>(ptr[AR_CTYPE]);
  W.Aval = ptr[AR_AVAL]; W.Dinv = ptr[AR_DINV]; W.Lsub = ptr[AR_LSUB];
  W.idx = reinterpret_cast<idx_t*>(ptr[AR_IDX]);
  W.Pval = ptr[AR_PVAL];
  const size_t np = P.tri_np;
  W.Lp = ptr[AR_LP];
  W.stage = kPlace == PLACE_SMEM ? nullptr : ptr[AR_STAGE];
  W.stage_stride = static_cast<int>((size_t(P.tri_bs) * P.tri_ld + 1) & ~size_t(1));
  double* bp = ptr[AR_SCRATCH];
  W.Dp = bp; bp += np * (np + 1);
  W.Dp2 = bp; bp += 2 * np * (np + 1);
  W.s_stride = static_cast<int>((size_t(P.tri_bs) * P.tri_ld + 1) & ~size_t(1));
  W.sp_stride = static_cast<int>((np * P.tri_bs + 1) & ~size_t(1));
  W.S = bp; bp += 2 * W.s_stride;
  W.Sp = bp; bp += 2 * W.sp_stride;
  W.xp = bp; bp += (np + 2) & ~size_t(1);
  W.piv = bp;
  W.Fb = nullptr;
  W.w = ptr[AR_W];
  W.D = ptr[AR_D]; W.E = ptr[AR_E]; W.dx = ptr[AR_DX]; W.dy = ptr[AR_DY];
}

struct Rho {
  double ineq, eq, inv_ineq, inv_eq;
  __device__ explicit Rho(double rho) : ineq(rho), eq(kRhoEqOverIneq * rho), inv_ineq(1.0 / rho), inv_eq(1.0 / (kRhoEqOverIneq * rho)) {}
  // ct == 1 ? a : (ct == -1 ? c : b) as two selects: written as a ternary the compiler rematerialises the equality
  // value inside a branch region per matrix entry / row (K assembly, update phase)
  __device__ static __forceinline__ double pick(double a, double b, double c, int ct) {
    double r;
    asm("{\n .reg .pred p, q;\n setp.eq.s32 p, %4, 1;\n setp.eq.s32 q, %4, -1;\n selp.f64 %0, %1, %2, p;\n selp.f64 %0, %3, %0, q;\n}"
        : "=&d"(r) : "d"(a), "d"(b), "d"(c), "r"(ct));
    return r;
  }
  __device__ __forceinline__ double of(signed char ct) const { return pick(eq, ineq, kRhoMin, ct); }
  __device__ __forceinline__ double inv(signed char ct) const { return pick(inv_eq, inv_ineq, 1.0 / kRhoMin, ct); }
};

// ---------------------------------------------------------------------------------------
// K -> factor storage: Dinv_k <- K_kk, Lsub_k <- K_{k,k-1}, Lp <- K_p., Dp <- K_pp
// entry (i, j) = [i == j] sigma + P_ij + sum_r rho_r A_ri A_rj  (sorted merge of two columns)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double k_entry(const PatternDev& P, const Work& W, const Rho& rho, double sigma, int i, int j) {
  double s = (i == j) ? sigma : 0.0;
  {
    const int e = P.p_colptr[j + 1];
    for (int k = P.p_colptr[j]; k < e; ++k)
      if (P.p_rowidx[k] == i) { s += W.Pval[k]; break; }
  }
  int ka = P.a_colptr[i], kc = P.a_colptr[j];
  const int ea = P.a_colptr[i + 1], ec = P.a_colptr[j + 1];
  if (ka < ea && kc < ec) {
    int ra = P.a_rowidx[ka], rc = P.a_rowidx[kc];
    while (true) {
      if (ra == rc) {
        s += rho.of(W.ctype[ra]) * W.Aval[ka] * W.Aval[kc];
        if (++ka >= ea || ++kc >= ec) break;
        ra = P.a_rowidx[ka]; rc = P.a_rowidx[kc];
      } else if (ra < rc) {
        if (++ka >= ea) break;
        ra = P.a_rowidx[ka];
      } else {
        if (++kc >= ec) break;
        rc = P.a_rowidx[kc];
      }
    }
  }
  return s;
}

// K assembly from the host-built program (PatternDev::kprog): zero the factor storage, then one
// thread per structurally non-zero element walks its runs of matching A entries.  Same summation
// order as the merging version below (sigma, P_ij, then products by ascending row).
__device__ inline void tri_assemble_program(const PatternDev& P, const Work& W, const Rho& rho, double sigma) {
  const int tid = threadIdx.x, T = blockDim.x;
  const int np = P.tri_np, bs = P.tri_bs, nb = P.tri_nb, ld = P.tri_ld, N = nb * bs;
  {
    const int nfac = nb * bs * ld;   // even (ld is even)
    double2* d2 = reinterpret_cast<double2*>(W.Dinv);
    double2* l2 = reinterpret_cast<double2*>(W.Lsub);
    const double2 z = make_double2(0.0, 0.0);
    for (int e = tid; e < nfac / 2; e += T) { d2[e] = z; l2[e] = z; }
    for (int e = tid; e < np * N; e += T) W.Lp[e] = 0.0;
    for (int e = tid; e < np * (np + 1); e += T) W.Dp[e] = 0.0;
  }
  __syncthreads();
  double* const arr[4] = {W.Dinv, W.Lsub, W.Lp, W.Dp};
  // The program lives in global memory (L2): an entry and its first run are two DEPENDENT loads, ~2 L2 round trips per
  // element if taken one at a time (the loop was bound by exactly that: 124 k cycles per QP at four CTAs per SM).  Four
  // elements per thread are fetched together -- four independent entry loads, then four independent run loads --
  // and computed in the old order, so every sum is bit-identical.
  constexpr int kBatch = 4;
  for (int e0 = tid; e0 < P.kprog_entries; e0 += kBatch * T) {
    KEntry ent[kBatch];
    KRun first[kBatch];
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const int e = e0 + u * T;
      ent[u] = P.kprog[e < P.kprog_entries ? e : e0];
    }
#pragma unroll
    for (int u = 0; u < kBatch; ++u) first[u] = P.kruns[ent[u].nruns > 0 ? ent[u].run_begin : 0];
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      if (e0 + u * T >= P.kprog_entries) continue;
      double s = ent[u].diag ? sigma : 0.0;
      if (ent[u].ppos >= 0) s += W.Pval[ent[u].ppos];
      for (int q = 0; q < ent[u].nruns; ++q) {
        const KRun run = q == 0 ? first[u] : P.kruns[ent[u].run_begin + q];
#pragma unroll 4
        for (int t = 0; t < run.len; ++t) {
          const int ka = run.ka + t, kc = run.kc + t;
          s += rho.of(W.ctype[run.row0 + t]) * W.Aval[ka] * W.Aval[kc];
        }
      }
      arr[ent[u].dest0 >> 30][ent[u].dest0 & 0x3fffffffu] = s;
      if (ent[u].dest1 != 0xffffffffu) arr[ent[u].dest1 >> 30][ent[u].dest1 & 0x3fffffffu] = s;
    }
  }
  __syncthreads();
}

__device__ inline void tri_assemble(const PatternDev& P, const Work& W, const Rho& rho, double sigma) {
  if (P.kprog_entries > 0) { tri_assemble_program(P, W, rho, sigma); return; }
  const int tid = threadIdx.x, T = blockDim.x;
  const int np = P.tri_np, bs = P.tri_bs, nb = P.tri_nb, ld = P.tri_ld, N = nb * bs;
  const int bb = bs * bs;
  // diagonal blocks: upper triangle computed, mirrored
  for (int e = tid; e < nb * bb; e += T) {
    const int k = e / bb, r = (e - k * bb) / bs, c = e - k * bb - r * bs;
    if (r > c) continue;
    const double v = k_entry(P, W, rho, sigma, np + k * bs + r, np + k * bs + c);
    double* Dk = W.Dinv + size_t(k) * bs * ld;
    Dk[r * ld + c] = v;
    Dk[c * ld + r] = v;
  }
  // sub-diagonal blocks K_{k,k-1}
  for (int e = tid; e < (nb - 1) * bb; e += T) {
    const int k = 1 + e / bb, r = (e - (k - 1) * bb) / bs, c = e - (k - 1) * bb - r * bs;
    W.Lsub[size_t(k) * bs * ld + r * ld + c] = k_entry(P, W, rho, sigma, np + k * bs + r, np + (k - 1) * bs + c);
  }
  // border rows
  for (int e = tid; e < np * N; e += T) {
    const int r = e / N, j = e - r * N;
    W.Lp[size_t(r) * N + j] = k_entry(P, W, rho, sigma, r, np + j);
  }
  for (int e = tid; e < np * np; e += T) {
    const int r = e / np, c = e - r * np;
    if (r > c) continue;
    const double v = k_entry(P, W, rho, sigma, r, c);
    W.Dp[r * (np + 1) + c] = v;
    W.Dp[c * (np + 1) + r] = v;
  }
  __syncthreads();
}

// in-place Gauss-Jordan inverse of an SPD block (no pivoting), executed by ONE warp
__device__ __forceinline__ void warp_invert(double* M, int bs, int ld, int lane) {
  for (int k = 0; k < bs; ++k) {
    const double ipiv = 1.0 / M[k * ld + k];
    __syncwarp();
    for (int c = lane; c < bs; c += 32) M[k * ld + c] = (c == k) ? ipiv : M[k * ld + c] * ipiv;
    __syncwarp();
    for (int idx = lane; idx < bs * bs; idx += 32) {
      const int r = idx / bs, c = idx - r * bs;
      if (r != k && c != k) M[r * ld + c] -= M[r * ld + k] * M[k * ld + c];
    }
    __syncwarp();
    for (int r = lane; r < bs; r += 32)
      if (r != k) M[r * ld + k] = -M[r * ld + k] * ipiv;
    __syncwarp();
  }
}

// in-place inverse of an SPD bs x bs block (Gauss-Jordan, no pivoting) by the WHOLE CTA, staged
// through a shared-memory scratch block (the block itself may live in the global slab).  Generic
// in bs; three barriers per pivot.  The exact-size one-warp version is in tri_fast.cuh.
__device__ inline void block_invert_coop(double* M, double* scratch, int bs, int ld) {
  const int tid = threadIdx.x, T = blockDim.x;
  const int bb = bs * bs;
  for (int e = tid; e < bs * ld; e += T) scratch[e] = M[e];
  __syncthreads();
  for (int k = 0; k < bs; ++k) {
    const double ipiv = 1.0 / scratch[k * ld + k];
    for (int e = tid; e < bb; e += T) {
      const int r = e / bs, c = e - r * bs;
      if (r != k && c != k) scratch[r * ld + c] -= scratch[r * ld + k] * (scratch[k * ld + c] * ipiv);
    }
    __syncthreads();
    for (int c = tid; c < bs; c += T) {
      if (c != k) {
        scratch[k * ld + c] *= ipiv;
        scratch[c * ld + k] *= -ipiv;
      }
    }
    if (tid == 0) scratch[k * ld + k] = ipiv;
    __syncthreads();
  }
  for (int e = tid; e < bs * ld; e += T) M[e] = scratch[e];
  __syncthreads();
}

// block LDL' of the bordered block-tridiagonal K held in the factor storage
__device__ inline void tri_factor(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int np = P.tri_np, bs = P.tri_bs, nb = P.tri_nb, ld = P.tri_ld, N = nb * bs;
  const int bb = bs * bs;
  for (int k = 0; k < nb; ++k) {
    double* Dk = W.Dinv + size_t(k) * bs * ld;
    if (k > 0) {
      double* Tk = W.Lsub + size_t(k) * bs * ld;               // K_{k,k-1}
      const double* Dm = W.Dinv + size_t(k - 1) * bs * ld;     // D_{k-1}^-1
      // S = K_{k,k-1} D_{k-1}^-1  (= L_k);  Sp = V_{k-1}
      for (int e = tid; e < bb; e += T) {
        const int r = e / bs, c = e - r * bs;
        double s = 0.0;
        for (int t = 0; t < bs; ++t) s += Tk[r * ld + t] * Dm[t * ld + c];
        W.S[r * ld + c] = s;
      }
      for (int e = tid; e < np * bs; e += T) {
        const int r = e / bs, c = e - r * bs;
        W.Sp[e] = W.Lp[size_t(r) * N + (k - 1) * bs + c];
      }
      __syncthreads();
      // D_k = K_kk - S K_{k,k-1}';  V_k = K_pk - V_{k-1} S';  L_{p,k-1} = V_{k-1} D_{k-1}^-1
      for (int e = tid; e < bb; e += T) {
        const int r = e / bs, c = e - r * bs;
        double s = 0.0;
        for (int t = 0; t < bs; ++t) s += W.S[r * ld + t] * Tk[c * ld + t];
        Dk[r * ld + c] -= s;
      }
      for (int e = tid; e < np * bs; e += T) {
        const int r = e / bs, c = e - r * bs;
        double s = 0.0, f = 0.0;
        for (int t = 0; t < bs; ++t) {
          const double v = W.Sp[r * bs + t];
          s += v * W.S[c * ld + t];
          f += v * Dm[t * ld + c];
        }
        W.Lp[size_t(r) * N + k * bs + c] -= s;
        W.Lp[size_t(r) * N + (k - 1) * bs + c] = f;
      }
      __syncthreads();
      // D_p -= V_{k-1} L_{p,k-1}';  L_k <- S
      for (int e = tid; e < np * np; e += T) {
        const int r = e / np, c = e - r * np;
        double s = 0.0;
        for (int t = 0; t < bs; ++t) s += W.Sp[r * bs + t] * W.Lp[size_t(c) * N + (k - 1) * bs + t];
        W.Dp[r * (np + 1) + c] -= s;
      }
      for (int e = tid; e < bb; e += T) {
        const int r = e / bs, c = e - r * bs;
        Tk[r * ld + c] = W.S[r * ld + c];
      }
    }
    block_invert_coop(Dk, W.S + W.s_stride, bs, ld);   // second scratch set: phase 3 may still read the first
  }
  // last border block, then D_p^-1
  if (np > 0) {
    const double* Dm = W.Dinv + size_t(nb - 1) * bs * ld;
    for (int e = tid; e < np * bs; e += T) {
      const int r = e / bs, c = e - r * bs;
      W.Sp[e] = W.Lp[size_t(r) * N + (nb - 1) * bs + c];
    }
    __syncthreads();
    for (int e = tid; e < np * bs; e += T) {
      const int r = e / bs, c = e - r * bs;
      double f = 0.0;
      for (int t = 0; t < bs; ++t) f += W.Sp[r * bs + t] * Dm[t * ld + c];
      W.Lp[size_t(r) * N + (nb - 1) * bs + c] = f;
    }
    __syncthreads();
    for (int e = tid; e < np * np; e += T) {
      const int r = e / np, c = e - r * np;
      double s = 0.0;
      for (int t = 0; t < bs; ++t) s += W.Sp[r * bs + t] * W.Lp[size_t(c) * N + (nb - 1) * bs + t];
      W.Dp[r * (np + 1) + c] -= s;
    }
    __syncthreads();
    if (warp == 0) warp_invert(W.Dp, np, np + 1, lane);
    __syncthreads();
  }
}

// Generic block sweep for any block size bs <= 64 (the exact-size code in tri_fast.cuh /
// tri_twisted.cuh covers bs = 16 and 20): four lanes per block row, the rows of a block spread
// over ceil(4 bs / 32) warps that meet at a named barrier after every stage; each lane keeps the
// next stage's slice of its row in registers (the factor may live in the global slab).
//   kColumn = false: y_k -= L_k y_{k-1}, k = 1..nb-1        kColumn = true: x_k -= L_{k+1}' x_{k+1}, k = nb-2..0
template <bool kColumn>
__device__ __forceinline__ void coop_sweep(const PatternDev& P, const Work& W, double* bx) {
  const int tid = threadIdx.x;
  const int bs = P.tri_bs, nb = P.tri_nb, ld = P.tri_ld;
  const int nthr = ((4 * bs + 31) / 32) * 32;   // participating threads (whole warps)
  if (tid >= nthr || nb < 2) return;
  const int row = tid >> 2, sub = tid & 3;
  const bool act = row < bs;
  const int rr = act ? row : 0;
  constexpr int kMaxPer = 16;                    // columns per lane: bs <= 64
  const int per = (bs + 3) >> 2;
  double cur[kMaxPer], nxt[kMaxPer];
  auto load = [&](double (&dst)[kMaxPer], int slot) {
    const double* base = W.Lsub + size_t(slot) * bs * ld;
#pragma unroll
    for (int i = 0; i < kMaxPer; ++i) {
      const int c = sub + 4 * i;
      dst[i] = (i < per && c < bs) ? (kColumn ? base[c * ld + rr] : base[rr * ld + c]) : 0.0;
    }
  };
  const int first = kColumn ? nb - 1 : 1, step = kColumn ? -1 : 1;
  load(cur, first);
  for (int t = 0; t < nb - 1; ++t) {
    const int slot = first + t * step;
    const int dstb = kColumn ? slot - 1 : slot, srcb = kColumn ? slot : slot - 1;
    if (t + 1 < nb - 1) load(nxt, slot + step);
    const double* src = bx + srcb * bs;
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int i = 0; i < kMaxPer; i += 2) {
      const int c0 = sub + 4 * i, c1 = sub + 4 * (i + 1);
      if (i < per && c0 < bs) s0 = fma(cur[i], src[c0], s0);
      if (i + 1 < per && c1 < bs) s1 = fma(cur[i + 1], src[c1], s1);
    }
    double sum = s0 + s1;
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    if (act && sub == 0) bx[dstb * bs + row] -= sum;
    asm volatile("bar.sync 4, %0;" ::"r"(nthr) : "memory");
#pragma unroll
    for (int i = 0; i < kMaxPer; ++i) cur[i] = nxt[i];
  }
}

// K x = b in place: b is [p | block 0 | ... | block nb-1]
__device__ inline void tri_solve(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  const int np = P.tri_np, bs = P.tri_bs, nb = P.tri_nb, ld = P.tri_ld, N = nb * bs;
  double* bx = W.b + np;
  OCP_B200_FINE_CLOCK(clk, W.phase);
  // forward sweep: y_k = b_k - L_k y_{k-1}
  coop_sweep<false>(P, W, bx);
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_FWD);
  // border: y_p = b_p - sum_k L_pk y_k  (a warp per border row), x_p = D_p^-1 y_p
  if (np > 0) {
    for (int r = warp; r < np; r += nw) {
      double s = 0.0;
      const double* row = W.Lp + size_t(r) * N;
#pragma unroll 8
      for (int j = lane; j < N; j += 32) s += row[j] * bx[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) W.xp[r] = W.b[r] - s;
    }
    __syncthreads();
    if (tid < np) {
      double s = 0.0;
      for (int c = 0; c < np; ++c) s += W.Dp[tid * (np + 1) + c] * W.xp[c];
      W.b[tid] = s;
    }
    __syncthreads();
  }
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BORDER);
  // diagonal: c_k = D_k^-1 y_k - L_pk' x_p   (in place: value computed, barrier, stored)
  const int Tb = (T / bs) * bs;   // whole blocks per pass: a pass never reads what it overwrites
  for (int base = 0; base < N; base += Tb) {
    const int j = tid < Tb ? base + tid : N;
    double v = 0.0;
    if (j < N) {
      const int k = j / bs, r = j - k * bs;
      const double* Dk = W.Dinv + size_t(k) * bs * ld + r * ld;
      const double* yk = bx + k * bs;
      double s0 = 0.0, s1 = 0.0;
      int c = 0;
#pragma unroll 4
      for (; c + 1 < bs; c += 2) { s0 += Dk[c] * yk[c]; s1 += Dk[c + 1] * yk[c + 1]; }
      if (c < bs) s0 += Dk[c] * yk[c];
      v = s0 + s1;
#pragma unroll 8
      for (int p = 0; p < np; ++p) v -= W.Lp[size_t(p) * N + j] * W.b[p];
    }
    __syncthreads();
    if (j < N) bx[j] = v;
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_DIAG);
  // backward sweep: x_k = c_k - L_{k+1}' x_{k+1}
  coop_sweep<true>(P, W, bx);
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BWD);
}

// K x = b in place with the factor STREAMED from the global slab (the problem is too large for the
// factor to stay on chip).  Every block of the factor is used exactly once per phase, so the three
// block phases -- forward sweep over L_1..L_{nb-1}, diagonal phase over D_0^-1..D_{nb-1}^-1, backward
// sweep over L_{nb-1}..L_1 -- pull their blocks through the shared-memory ring (block_ring.cuh: bulk
// copies, ring_slots blocks in flight) and read them from shared memory, which also makes the
// transposed access of the backward sweep conflict-free instead of uncoalesced.  Four lanes per block
// row as in coop_sweep; one named barrier per stage.  kBS > 0: compile-time block size (pitch kBS + 2),
// every loop unrolled and all shared-memory loads of a stage issued before its first FMA; kBS == 0:
// any block size.
template <int kBS>
__device__ inline void tri_solve_stream(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  const int np = P.tri_np, nb = P.tri_nb;
  const int bs = kBS > 0 ? kBS : P.tri_bs, ld = kBS > 0 ? kBS + 2 : P.tri_ld, N = nb * bs;
  // fields are copied into locals: W and P live in the caller's frame and the "memory" clobbers of the
  // barrier / bulk-copy instructions would turn each later use into a reload through local memory
  // b and the ring slots are in shared memory whenever this function runs (the kernel checks the placement mask
  // before it sets ring_slots): both pointers are re-derived from the dynamic shared-memory symbol, so that the
  // sweeps load with LDS and 32-bit addresses instead of generic loads
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* const sm0 = reinterpret_cast<double*>(smem_raw);
  double* const wb = sm0 + (W.b - sm0);
  double* const bx = wb + np;
  const double* const Lsub = W.Lsub;
  const double* const Dinv = W.Dinv;
  const double* const Lp = W.Lp;
  double* const xp = W.xp;
  const double* const Dp = W.Dp;
  double* const Dp2 = W.Dp2;
  double* const stage = sm0 + (W.stage - sm0);
  double* const Sbuf = sm0 + (W.S - sm0);   // (a ring slot only when the scratch is in shared memory too)
  unsigned long long* const ring_bar = W.ring_bar;
  unsigned* const ring_phase = W.ring_phase;
  const int s_stride = W.s_stride, stage_slots = P.stage_slots;
  const int R = W.ring_slots, stride = W.stage_stride;
  const uint32_t bytes = static_cast<uint32_t>(bs * ld * sizeof(double));
  const int nthr = ((4 * bs + 31) / 32) * 32;   // participating threads (whole warps)
  const int row = tid >> 2, sub = tid & 3;
  const bool part = tid < nthr, act = part && row < bs;
  // the warp after the compute warps only issues the bulk copies (an issue costs the issuing warp ~300
  // cycles, which would otherwise sit on the critical path of every stage); it joins the named barrier of
  // the stages, so it knows when a slot is free.  Without a spare warp thread 0 issues.
  const bool has_issuer = nthr + 32 <= T;
  const bool issue_thread = has_issuer ? tid == nthr : tid == 0;
  const bool in_loop = part || (has_issuer && tid < nthr + 32);
  const int nbar = has_issuer ? nthr + 32 : nthr;
  const int rr = act ? row : 0;
  constexpr int kPer = kBS > 0 ? (kBS + 3) / 4 : 16;   // columns per lane (bs <= 64)
  uint32_t ph = ring_phase[0];   // identical in every participating thread
  OCP_B200_FINE_CLOCK(clk, W.phase);

  // The three block phases form ONE stream of G = 2 (nb - 1) + nb blocks, so the ring never drains
  // between them (and keeps filling during the border phase): stream position g -> block address.
  // Ring slots: the staging area, then the two block-sized scratch buffers of the factorisation.
  // (compile-time block size: the diagonal phase is not part of the stream -- all threads read their D_k^-1 rows
  // straight from the slab, see below -- and the ring goes from the forward blocks to the backward blocks)
#ifndef OCP_B200_RING_DIAG
#define OCP_B200_RING_DIAG 0   // 1: the diagonal phase through the ring as well (A/B measurements)
#endif
  constexpr bool kParallelDiag = kBS > 0 && !OCP_B200_RING_DIAG;
  const int G = 2 * (nb - 1) + (kParallelDiag ? 0 : nb);
  const size_t blk_doubles = size_t(bs) * ld;
  auto gaddr = [&](int g) -> const double* {
    if (g < nb - 1) return Lsub + size_t(1 + g) * blk_doubles;
    g -= nb - 1;
    if (!kParallelDiag) {
      if (g < nb) return Dinv + size_t(g) * blk_doubles;
      g -= nb;
    }
    return Lsub + size_t(nb - 1 - g) * blk_doubles;
  };
  auto slot_ptr = [&](int sl) -> double* {
    return sl < stage_slots ? stage + sl * stride : Sbuf + (sl - stage_slots) * s_stride;
  };
  if (issue_thread)
    for (int i = 0; i < R && i < G; ++i) ring_issue(slot_ptr(i), gaddr(i), bytes, ring_bar + i);
  int g = 0, s = 0;   // stream position, ring slot
  auto advance = [&]() {   // after the stage's barrier: the slot is free, request the block R positions ahead
    if (issue_thread && g + R < G) ring_issue(slot_ptr(s), gaddr(g + R), bytes, ring_bar + s);
    ++g;
    s = s + 1 == R ? 0 : s + 1;
  };
  // sum over this lane's columns c = sub, sub + 4, ... of M[rr][c] src[c] (or M[c][rr] src[c]),
  // combined over the four lanes of the row
  auto block_dot = [&](const double* blk, const double* src, bool column) {
    double mv[kPer], sv[kPer];
    const double* mp = column ? blk + rr : blk + rr * ld;
    const int ms = column ? ld : 1;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int c = sub + 4 * i;
      const bool ok = c < bs;
      mv[i] = ok ? mp[c * ms] : 0.0;
      sv[i] = ok ? src[c] : 0.0;
    }
    double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
    for (int i = 0; i < kPer; i += 3) {
      s0 = fma(mv[i], sv[i], s0);
      if (i + 1 < kPer) s1 = fma(mv[i + 1], sv[i + 1], s1);
      if (i + 2 < kPer) s2 = fma(mv[i + 2], sv[i + 2], s2);
    }
    double sum = (s0 + s1) + s2;
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    return sum;
  };

  // forward sweep: y_k = b_k - L_k y_{k-1}, k = 1..nb-1
  if (in_loop) {
    for (int t = 0; t < nb - 1; ++t) {
      if (part) {
        ring_wait(ring_bar + s, (ph >> s) & 1u);
        ph ^= 1u << s;
        const double old = (act && sub == 0) ? bx[(t + 1) * bs + row] : 0.0;
        const double sum = block_dot(slot_ptr(s), bx + t * bs, false);
        if (act && sub == 0) bx[(t + 1) * bs + row] = old - sum;
      }
      asm volatile("bar.sync 4, %0;" ::"r"(nbar) : "memory");
      advance();
    }
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_FWD);

  // border: y_p = b_p - sum_k L_pk y_k.  L_p [np x N] is streamed once: every thread owns a strided set
  // of column pairs and keeps eight border rows' partial sums, all eight 16-byte loads of a column pair
  // issued together; the warps' sums meet in shared memory in a fixed order.  Then x_p = D_p^-1 y_p.
  if (np > 0) {
    const bool vec = (N & 1) == 0 && (reinterpret_cast<unsigned long long>(bx) & 15ULL) == 0ULL &&
                     (reinterpret_cast<unsigned long long>(Lp) & 15ULL) == 0ULL;
    double* part_sums = Dp2;   // factor scratch, free during a solve: [warp][8]
    const bool wide_border = 2 * np * (np + 1) >= nw * 8;
    if (!wide_border) {   // small border: a warp per row
      for (int r = warp; r < np; r += nw) {
        double sacc = 0.0;
        const double* rowp = Lp + size_t(r) * N;
#pragma unroll 8
        for (int j = lane; j < N; j += 32) sacc += rowp[j] * bx[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (lane == 0) xp[r] = wb[r] - sacc;
      }
      __syncthreads();
    }
    for (int r0 = 0; wide_border && r0 < np; r0 += 8) {
      double acc[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      if (vec) {
        const double2* y2 = reinterpret_cast<const double2*>(bx);
#pragma unroll 2
        for (int j = tid; j < N / 2; j += T) {
          double2 v[8];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            v[q] = r0 + q < np ? reinterpret_cast<const double2*>(Lp + size_t(r0 + q) * N)[j] : make_double2(0.0, 0.0);
          const double2 y = y2[j];
#pragma unroll
          for (int q = 0; q < 8; ++q) acc[q] = fma(v[q].x, y.x, fma(v[q].y, y.y, acc[q]));
        }
      } else {
        for (int j = tid; j < N; j += T) {
          const double y = bx[j];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (r0 + q < np) acc[q] = fma(Lp[size_t(r0 + q) * N + j], y, acc[q]);
        }
      }
#pragma unroll
      for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
        if (lane == 0) part_sums[warp * 8 + q] = acc[q];
      }
      __syncthreads();
      if (tid < 8 && r0 + tid < np) {
        double sacc = 0.0;
        for (int w = 0; w < nw; ++w) sacc += part_sums[w * 8 + tid];
        xp[r0 + tid] = wb[r0 + tid] - sacc;
      }
      __syncthreads();
    }
    if (tid < np) {
      double sacc = 0.0;
      for (int c = 0; c < np; ++c) sacc += Dp[tid * (np + 1) + c] * xp[c];
      wb[tid] = sacc;
    }
    __syncthreads();
  }
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BORDER);

  // diagonal phase: c_k = D_k^-1 y_k - L_pk' x_p.  Compile-time block size: one row per thread and pass, whole
  // blocks per pass (a pass never reads what it overwrites), every load of a row issued before its first FMA --
  // the phase runs at the rate the slab delivers D^-1 and L_p to ALL threads instead of one ring stage per block.
  // Any block size: block by block through the ring; the L_p values of the next block are requested before the
  // current block is multiplied.
  if constexpr (kParallelDiag) {
    // four lanes per row (9 of 36 columns each: few enough registers that every load of a pass is in flight
    // before the first FMA -- this kernel runs 768 threads at 80 registers), T / 4 rows per pass, whole blocks
    static_assert(kBS % 4 == 0, "columns split over four lanes");
    constexpr int kPerD = kBS / 4, kMaxLp = 8;   // border rows per lane: np <= 32, else a loop
    const int rows_pass = ((T >> 2) / kBS) * kBS;
    const int prow = tid >> 2, psub = tid & 3;
    for (int base = 0; base < N; base += rows_pass) {
      const int j = prow < rows_pass ? base + prow : N;
      const bool have = j < N;
      const int jj = have ? j : 0;   // (clamped: unconditional loads, result dropped)
      const int k = jj / kBS, r = jj - k * kBS;
      const double* drow = Dinv + size_t(k) * blk_doubles + r * ld + psub;
      const double* yk = bx + k * kBS + psub;
      double mv[kPerD], sv[kPerD], lv[kMaxLp], xv[kMaxLp];
#pragma unroll
      for (int i = 0; i < kPerD; ++i) mv[i] = drow[4 * i];
#pragma unroll
      for (int i = 0; i < kMaxLp; ++i) {
        const int pp = psub + 4 * i;
        lv[i] = Lp[size_t(pp < np ? pp : 0) * N + jj];
      }
#pragma unroll
      for (int i = 0; i < kPerD; ++i) sv[i] = yk[4 * i];
#pragma unroll
      for (int i = 0; i < kMaxLp; ++i) {
        const int pp = psub + 4 * i;
        const double x = wb[pp < np ? pp : 0];
        xv[i] = pp < np ? x : 0.0;
      }
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
      for (int i = 0; i < kPerD; i += 3) {
        s0 = fma(mv[i], sv[i], s0);
        if (i + 1 < kPerD) s1 = fma(mv[i + 1], sv[i + 1], s1);
        if (i + 2 < kPerD) s2 = fma(mv[i + 2], sv[i + 2], s2);
      }
      double c0 = 0.0, c1 = 0.0;
#pragma unroll
      for (int i = 0; i < kMaxLp; i += 2) { c0 = fma(lv[i], xv[i], c0); c1 = fma(lv[i + 1], xv[i + 1], c1); }
      double v = ((s0 + s1) + s2) - (c0 + c1);
      if (np > 4 * kMaxLp)
        for (int pp = psub + 4 * kMaxLp; pp < np; pp += 4) v = fma(-Lp[size_t(pp) * N + jj], wb[pp], v);
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      __syncthreads();
      if (have && psub == 0) bx[j] = v;
    }
  } else if (in_loop) {
    const int count = nb;
    constexpr int kMaxLp = 8;   // border rows per lane: np <= 32
    const bool lp_regs = np <= 4 * kMaxLp;
    double lpn[kMaxLp] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    auto fetch_lp = [&](int k) {
#pragma unroll
      for (int i = 0; i < kMaxLp; ++i) {
        const int p = sub + 4 * i;
        lpn[i] = (act && p < np) ? Lp[size_t(p) * N + k * bs + row] : 0.0;
      }
    };
    if (lp_regs) fetch_lp(0);
    double xpv[kMaxLp];
#pragma unroll
    for (int i = 0; i < kMaxLp; ++i) xpv[i] = (lp_regs && sub + 4 * i < np) ? wb[sub + 4 * i] : 0.0;
    for (int k = 0; k < count; ++k) {
      double corr = 0.0, corr1 = 0.0;
      if (lp_regs) {
#pragma unroll
        for (int i = 0; i < kMaxLp; i += 2) { corr = fma(lpn[i], xpv[i], corr); corr1 = fma(lpn[i + 1], xpv[i + 1], corr1); }
        corr += corr1;
        if (k + 1 < count) fetch_lp(k + 1);
      } else if (act) {
        for (int p = sub; p < np; p += 4) corr = fma(Lp[size_t(p) * N + k * bs + row], wb[p], corr);
      }
      double v = 0.0;
      if (part) {
        ring_wait(ring_bar + s, (ph >> s) & 1u);
        ph ^= 1u << s;
        v = block_dot(slot_ptr(s), bx + k * bs, false);
        corr += __shfl_xor_sync(0xffffffffu, corr, 1);
        corr += __shfl_xor_sync(0xffffffffu, corr, 2);
      }
      asm volatile("bar.sync 4, %0;" ::"r"(nbar) : "memory");   // every row has read y_k
      if (act && sub == 0) bx[k * bs + row] = v - corr;
      advance();
    }
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_DIAG);

  // backward sweep: x_k = c_k - L_{k+1}' x_{k+1}, k = nb-2..0
  if (in_loop) {
    for (int t = 0; t < nb - 1; ++t) {
      const int blkid = nb - 1 - t;
      if (part) {
        ring_wait(ring_bar + s, (ph >> s) & 1u);
        ph ^= 1u << s;
        const double old = (act && sub == 0) ? bx[(blkid - 1) * bs + row] : 0.0;
        const double sum = block_dot(slot_ptr(s), bx + blkid * bs, true);
        if (act && sub == 0) bx[(blkid - 1) * bs + row] = old - sum;
      }
      asm volatile("bar.sync 4, %0;" ::"r"(nbar) : "memory");
      advance();
    }
  }
  if (tid == 0) ring_phase[0] = ph;
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BWD);
}

// Streamed solve against the TWISTED factor of tri_twisted.cuh (blocks eliminated from both ends, meeting
// at block mid = nb / 2): two thread groups, four lanes per block row each, run the two chains of the
// forward sweep, split the diagonal phase between them and run the two chains of the backward sweep; each
// group pulls ITS sequence of factor blocks through its own ring (half of the staging area), as one stream
// that keeps filling across the phases and during the border product.  Used when the factor is slab-resident
// and a block row is too long for one lane (tri_twisted.cuh: one warp per chain, one lane per row, costs
// ~900 cycles per stage for 20 columns; this form ~300).
template <int kBS>
__device__ __noinline__ void tri_solve_stream_twisted(const PatternDev& P, const Work& W) {
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  // every field used below is copied into a local first: W and P live in the caller's frame, and the
  // "memory" clobbers of the barrier / bulk-copy instructions would make each later use a reload
  // through local memory (an L2 round trip when shared memory leaves almost no L1)
  const int np = P.tri_np, nb = P.tri_nb;
  constexpr int bs = kBS, ld = kBS + 2;
  const int N = nb * bs, mid = nb / 2;
  // b and the ring are in shared memory on this path (PLACE_BIG): re-derive both pointers from the dynamic
  // shared-memory symbol, so that the sweeps load with LDS and 32-bit addresses instead of generic loads
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double* const sm0 = reinterpret_cast<double*>(smem_raw);
  double* const wb = sm0 + (W.b - sm0);
  double* const bx = wb + np;
  const double* const Lsub = W.Lsub;
  const double* const Dinv = W.Dinv;
  const double* const Lp = W.Lp;
  double* const xp = W.xp;
  double* const piv = W.piv;
  const double* const Dp = W.Dp;
  unsigned* const ring_phase = W.ring_phase;
  const int R = W.ring_slots, stride = W.stage_stride;
  constexpr uint32_t bytes = bs * ld * sizeof(double);
  constexpr int nthr = ((4 * bs + 31) / 32) * 32;   // threads per group (whole warps)
  const int GT = T / 2, grp = tid >= GT ? 1 : 0, gt = tid - grp * GT;
  const int row = gt >> 2, sub = gt & 3;
  // the warp after a group's compute warps only issues the bulk copies: an issue costs the issuing warp
  // ~300 cycles, which would otherwise sit on the critical path of every stage; it joins the group's
  // named barrier, so it knows when a slot is free
  const bool part = gt < nthr, act = part && row < bs;
  const bool issuer = gt >= nthr && gt < nthr + 32, in_grp = part || issuer;
  constexpr int nbar = nthr + 32;
  const int rr = act ? row : 0;
  constexpr int kPer = (kBS + 3) / 4;
  uint32_t ph = ring_phase[grp];
  double* ring = sm0 + (W.stage - sm0) + grp * R * stride;
  unsigned long long* bars = W.ring_bar + grp * kMaxRing;
  const int bar_id = 1 + grp;
  OCP_B200_FINE_CLOCK(clk, W.phase);

  // this group's block sequence: forward chain, (group 0: the two joining blocks,) backward chain.  The diagonal
  // phase is not a chain: all threads read their D_k^-1 rows straight from the slab (below) while the ring
  // already fills with the first blocks of the backward chain.
  const int n_fwd = grp == 0 ? mid - 1 : nb - 2 - mid;
  const int n_join = grp == 0 ? 2 : 0;
  const int n_bwd = grp == 0 ? mid : nb - 1 - mid;
  const int G = n_fwd + n_join + n_bwd;
  constexpr size_t blk_doubles = size_t(bs) * ld;
  auto gaddr = [&](int g) -> const double* {
    if (g < n_fwd) return Lsub + size_t(grp == 0 ? 1 + g : nb - 1 - g) * blk_doubles;
    g -= n_fwd;
    if (g < n_join) return Lsub + size_t(mid + g) * blk_doubles;
    g -= n_join;
    return Lsub + size_t(grp == 0 ? mid - g : mid + 1 + g) * blk_doubles;
  };
  if (issuer && lane == 0)
    for (int i = 0; i < R && i < G; ++i) ring_issue(ring + i * stride, gaddr(i), bytes, bars + i);
  int g = 0, s = 0;
  auto advance = [&]() {
    if (issuer && lane == 0 && g + R < G) ring_issue(ring + s * stride, gaddr(g + R), bytes, bars + s);
    ++g;
    s = s + 1 == R ? 0 : s + 1;
  };
  auto block_dot = [&](const double* blk, const double* src, bool column) {
    double mv[kPer], sv[kPer];
    const double* mp = column ? blk + rr : blk + rr * ld;
    const int ms = column ? ld : 1;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int c = sub + 4 * i;
      const bool ok = c < bs;
      mv[i] = ok ? mp[c * ms] : 0.0;
      sv[i] = ok ? src[c] : 0.0;
    }
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int i = 0; i < kPer; i += 2) {
      s0 = fma(mv[i], sv[i], s0);
      if (i + 1 < kPer) s1 = fma(mv[i + 1], sv[i + 1], s1);
    }
    double sum = s0 + s1;
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    return sum;
  };
  // one sweep stage: dst block -= M src block (M row-wise in the forward sweeps, transposed in the backward ones)
#ifdef OCP_B200_SWEEP_PROBE   // stage anatomy (thread 0): wait for the block / product / barrier / next issue
  PhaseClock pclk(W.phase);
#define OCP_B200_PROBE_LAP(slot) pclk.lap(slot)
#else
#define OCP_B200_PROBE_LAP(slot)
#endif
  auto sweep = [&](int dstb, int srcb, bool column) {
    OCP_B200_PROBE_LAP(OCP_B200_PHASE_SOLVE_BWD);
    if (part) {
      ring_wait(bars + s, (ph >> s) & 1u);
      ph ^= 1u << s;
      OCP_B200_PROBE_LAP(OCP_B200_PHASE_FACTOR_INVERT);
      const double old = (act && sub == 0) ? bx[dstb * bs + row] : 0.0;
      const double sum = block_dot(ring + s * stride, bx + srcb * bs, column);
      if (act && sub == 0) bx[dstb * bs + row] = old - sum;
      OCP_B200_PROBE_LAP(OCP_B200_PHASE_FACTOR_STEP);
    }
    asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nbar) : "memory");
    OCP_B200_PROBE_LAP(OCP_B200_PHASE_SOLVE_DIAG);
    advance();
    OCP_B200_PROBE_LAP(OCP_B200_PHASE_SOLVE_BORDER);
  };

  // forward: top chain y_k = b_k - L_k y_{k-1} (k = 1..mid-1), bottom chain y_k = b_k - U_k y_{k+1} (k = nb-2..mid+1)
  if (in_grp) {
    if (grp == 0) for (int i = 0; i < n_fwd; ++i) sweep(1 + i, i, false);
    else for (int i = 0; i < n_fwd; ++i) sweep(nb - 2 - i, nb - 1 - i, false);
  }
  __syncthreads();
  if (in_grp && grp == 0) {   // both contributions to block mid
    sweep(mid, mid - 1, false);
    sweep(mid, mid + 1, false);
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_FWD);

  // border: y_p = b_p - sum_k L_pk y_k with TPR threads per border row (one or two batches of eight
  // loads each, so a slab-resident L_p costs one or two round trips), then x_p = D_p^-1 y_p
  if (np > 0) {
    int TPR = 32;
    while (TPR * 2 * np <= T && (TPR * 2 / 32) * np <= 64 && TPR < 256) TPR *= 2;
    const int wpr = TPR / 32;
    if (np * 32 <= T) {
      const int r = tid / TPR, q = tid - r * TPR;
      const bool have = r < np;
      const double* rowp = Lp + size_t(have ? r : 0) * N;
      double s0 = 0.0, s1 = 0.0;
      for (int j0 = q; j0 < N; j0 += 8 * TPR) {
        double lv[8], yv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int j = j0 + TPR * u;
          const bool ok = have && j < N;
          lv[u] = ok ? rowp[j] : 0.0;
          yv[u] = ok ? bx[j] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; u += 2) { s0 = fma(lv[u], yv[u], s0); s1 = fma(lv[u + 1], yv[u + 1], s1); }
      }
      double sacc = s0 + s1;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
      if (have && lane == 0) piv[warp] = sacc;   // warp = r * wpr + (warp within the row)
      __syncthreads();
      if (tid < np) {
        double t = 0.0;
        for (int w = 0; w < wpr; ++w) t += piv[tid * wpr + w];
        xp[tid] = wb[tid] - t;
      }
    } else {
      const int nw = T >> 5;
      for (int r = warp; r < np; r += nw) {
        double sacc = 0.0;
        const double* rowp = Lp + size_t(r) * N;
#pragma unroll 8
        for (int j = lane; j < N; j += 32) sacc += rowp[j] * bx[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
        if (lane == 0) xp[r] = wb[r] - sacc;
      }
    }
    __syncthreads();
    if (tid < np) {
      double sacc = 0.0;
      for (int c = 0; c < np; ++c) sacc += Dp[tid * (np + 1) + c] * xp[c];
      wb[tid] = sacc;
    }
    __syncthreads();
  }
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BORDER);

  // diagonal phase: c_k = D_k^-1 y_k - L_pk' x_p, one row per thread and pass, whole blocks per pass (a pass never
  // reads what it overwrites); every load of a row is issued before its first FMA (one L2 round trip per pass
  // instead of one ring stage per block: 50 dependent stages -> 3 passes for the H = 200 cart-pole)
  {
    const int Tb = (T / bs) * bs;
    for (int base = 0; base < N; base += Tb) {
      const int j = tid < Tb ? base + tid : N;
      double v = 0.0;
      if (j < N) {
        const int k = j / bs, r = j - k * bs;
        const double2* d2 = reinterpret_cast<const double2*>(Dinv + size_t(k) * blk_doubles + r * ld);
        const double* yk = bx + k * bs;
        double dr[bs];
#pragma unroll
        for (int t = 0; t < bs / 2; ++t) { const double2 x = d2[t]; dr[2 * t] = x.x; dr[2 * t + 1] = x.y; }
        double corr = 0.0, corr1 = 0.0;
        if (np == 4) {
          double l0 = Lp[j], l1 = Lp[size_t(N) + j], l2 = Lp[2 * size_t(N) + j], l3 = Lp[3 * size_t(N) + j];
          corr = fma(l0, wb[0], fma(l2, wb[2], 0.0));
          corr1 = fma(l1, wb[1], fma(l3, wb[3], 0.0));
        } else {
          for (int p = 0; p < np; ++p) corr = fma(Lp[size_t(p) * N + j], wb[p], corr);
        }
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
        for (int t = 0; t < bs; t += 4) {
          s0 = fma(dr[t], yk[t], s0); s1 = fma(dr[t + 1], yk[t + 1], s1);
          s2 = fma(dr[t + 2], yk[t + 2], s2); s3 = fma(dr[t + 3], yk[t + 3], s3);
        }
        v = ((s0 + s1) + (s2 + s3)) - (corr + corr1);
      }
      __syncthreads();
      if (j < N) bx[j] = v;
    }
  }
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_DIAG);

  // backward, from block mid outwards: x_k = c_k - L_{k+1}' x_{k+1} (k = mid-1..0), x_k = c_k - U_{k-1}' x_{k-1} (k = mid+1..nb-1)
  if (in_grp) {
    if (grp == 0) for (int j = 0; j < n_bwd; ++j) sweep(mid - 1 - j, mid - j, true);
    else for (int j = 0; j < n_bwd; ++j) sweep(mid + 1 + j, mid + j, true);
  }
  if (part && gt == 0) ring_phase[grp] = ph;
  __syncthreads();
  OCP_B200_FINE_LAP(clk, OCP_B200_PHASE_SOLVE_BWD);
}

}  // namespace direct
}  // namespace ocpb200
#include "tri_fast.cuh"
#include "tri_twisted.cuh"
namespace ocpb200 {
namespace direct {

// block sizes with exact-size (compile-time) factorisation and sweeps: tri_fast.cuh / tri_twisted.cuh
__device__ __forceinline__ bool exact_block_code(const PatternDev& P) {
  return (P.tri_bs == 16 && P.tri_ld == 18) || (P.tri_bs == 20 && P.tri_ld == 22);
}

// block-size dispatch (uniform across the CTA)
template <int kPlace>
__device__ __forceinline__ void factor_dispatch(const PatternDev& P, const Work& W) {
  // exact-size code assumes the pitch tri_ld == bs + 2 (what the host sets for even block sizes)
  if (P.tri_bs == 16 && P.tri_ld == 18) tri_factor_twisted<16>(P, W);
  else if (P.tri_bs == 20 && P.tri_ld == 22) tri_factor_twisted<20>(P, W);
  else tri_factor(P, W);
  if (W.ring_slots > 0) {
    // the sweeps read the new factor through the async proxy (bulk copies): order the generic-proxy
    // stores of the factorisation before them
    asm volatile("fence.proxy.async.global;" ::: "memory");
    __syncthreads();
  }
}
template <int kPlace>
__device__ __forceinline__ void solve_dispatch(const PatternDev& P, const Work& W) {
  if (P.tri_bs == 16 && P.tri_ld == 18) tri_solve_twisted<16>(P, W);
  else if (P.tri_bs == 20 && P.tri_ld == 22) {
    if (kPlace == PLACE_BIG && W.ring_slots >= 2 && P.tri_nb >= 4 && 2 * (((4 * 20 + 31) / 32) * 32 + 32) <= int(blockDim.x)) {
      if constexpr (kPlace == PLACE_BIG) tri_solve_stream_twisted<20>(P, W);
    } else {
      tri_solve_twisted<20>(P, W);
    }
  }
  else if (kPlace == PLACE_MIXED && W.ring_slots > 0) {   // only the mixed placement streams generic blocks
    if constexpr (kPlace == PLACE_MIXED) {
      if (P.tri_bs == 36 && P.tri_ld == 38) tri_solve_stream<36>(P, W);
      else if (P.tri_bs == 24 && P.tri_ld == 26) tri_solve_stream<24>(P, W);
      else tri_solve_stream<0>(P, W);
    }
  }
  else tri_solve(P, W);
}

// ---------------------------------------------------------------------------------------
// one QP, solved by the whole CTA
// ---------------------------------------------------------------------------------------
template <int kPlace>
__device__ inline void solve_instance(const PatternDev& P, const ocp_b200_settings& S, const SolveArgs& A,
                                      const Work& W, Reducer& R, int inst, QpResult& out) {
  const int tid = threadIdx.x, T = blockDim.x;
  const int n = P.n, m = P.m;
  const double sigma = S.sigma, relax = S.relax;
  PhaseClock clk(A.phase);
  const_cast<Work&>(W).phase = A.phase;

  // ---- load (osqp_setup copies its inputs): values, q, bounds clamped to +-1e30 ------------
  {
    const double* hv = A.h_vals + size_t(inst) * A.ld_h;
    const double* av = A.a_vals + size_t(inst) * A.ld_a;
    const double* qv = A.q + size_t(inst) * A.ld_n;
    const double* lv = A.l + size_t(inst) * A.ld_m;
    const double* uv = A.u + size_t(inst) * A.ld_m;
    for (int k = tid; k < P.nnz_a; k += T) W.Aval[k] = av[k];
    for (int k = tid; k < P.nnz_p; k += T) { const int s = P.p_src[k]; W.Pval[k] = s >= 0 ? hv[s] : 0.0; }
    for (int j = tid; j < n; j += T) { W.q[j] = qv[j]; W.D[j] = 1.0; W.x[j] = 0.0; }
    double bad[1] = {0.0};
    for (int i = tid; i < m; i += T) {
      const double lo = lv[i], hi = uv[i];
      if (lo > hi) bad[0] = 1.0;
      W.l[i] = fmax(lo, -kInfty);
      W.u[i] = fmin(hi, kInfty);
      W.E[i] = 1.0; W.z[i] = 0.0; W.y[i] = 0.0; W.w[i] = 0.0;
    }
    block_reduce<1, true>(bad, R);
    if (bad[0] > 0.0) {  // osqp_setup rejects l > u; the reference then adds no usable step
      out = QpResult{OCP_B200_QP_UNSOLVED, 0, 0, 0, 0, 0.0, 0.0, S.rho};
      return;
    }
  }

  clk.lap(OCP_B200_PHASE_LOAD);
  // ---- Ruiz equilibration (scale_data): D, E, c;  scratch: b (n), dy (m), x (n), w (n) --------
  // The column norms of pass k+1 are by-products of the scaling of pass k: the scaled A column is in
  // hand when it is written (x keeps its inf-norm), and the P column norm is the one computed for the
  // cost normalisation times the cost factor ct (rounding is monotone, so the maximum commutes with
  // the multiplication bit for bit).  Only the first pass reads the matrices for its column norms.
  double c = 1.0;
  for (int pass = 0; pass < S.scaling_iters; ++pass) {
    for (int j = tid; j < n; j += T) {
      double dn = 0.0;
      if (pass == 0) {
#pragma unroll 4
        for (int k = P.p_colptr[j]; k < P.p_colptr[j + 1]; ++k) dn = fmax(dn, fabs(W.Pval[k]));
#pragma unroll 4
        for (int k = P.a_colptr[j]; k < P.a_colptr[j + 1]; ++k) dn = fmax(dn, fabs(W.Aval[k]));
      } else {
        dn = fmax(W.w[j], W.x[j]);
      }
      W.b[j] = 1.0 / sqrt(limit_scaling(dn));
    }
    for (int i = tid; i < m; i += T) {
      double en = 0.0;
#pragma unroll 4
      for (int k = P.a_rowptr[i]; k < P.a_rowptr[i + 1]; ++k) en = fmax(en, fabs(W.Aval[P.a_perm[k]]));
      W.dy[i] = 1.0 / sqrt(limit_scaling(en));
    }
    __syncthreads();
    double red[2] = {0.0, 0.0};  // sum of P column norms, max |q|
    for (int j = tid; j < n; j += T) {
      const double dj = W.b[j];
      double cn = 0.0, an = 0.0;
      for (int k = P.p_colptr[j]; k < P.p_colptr[j + 1]; ++k) {
        const double v = W.Pval[k] * W.b[P.p_rowidx[k]] * dj;
        W.Pval[k] = v;
        cn = fmax(cn, fabs(v));
      }
#pragma unroll 4
      for (int k = P.a_colptr[j]; k < P.a_colptr[j + 1]; ++k) {
        const double v = W.Aval[k] * (W.dy[P.a_rowidx[k]] * dj);
        W.Aval[k] = v;
        an = fmax(an, fabs(v));
      }
      W.x[j] = an;      // inf-norm of the scaled A column
      W.w[j] = cn;      // inf-norm of the scaled P column, before the cost factor
      const double qj = W.q[j] * dj;
      W.q[j] = qj;
      W.D[j] *= dj;
      red[0] += cn;
      red[1] = fmax(red[1], fabs(qj));
    }
    for (int i = tid; i < m; i += T) W.E[i] *= W.dy[i];
    double sum[1] = {red[0]}, mx[1] = {red[1]};
    block_reduce<1, false>(sum, R);
    block_reduce<1, true>(mx, R);
    const double ct = 1.0 / limit_scaling(fmax(sum[0] / double(n), limit_scaling(mx[0])));
    for (int k = tid; k < P.nnz_p; k += T) W.Pval[k] *= ct;
    for (int j = tid; j < n; j += T) { W.q[j] *= ct; W.w[j] *= ct; }
    c *= ct;
    __syncthreads();
  }
  for (int j = tid; j < n; j += T) { W.x[j] = 0.0; W.w[j] = 0.0; }   // back to the cold start
  const double cinv = 1.0 / c;

  // ---- scaled bounds, constraint types (set_rho_vec) ------------------------------------------
  double rho = fmin(fmax(S.rho, kRhoMin), kRhoMax);
  for (int i = tid; i < m; i += T) {
    const double lo = W.l[i] * W.E[i], hi = W.u[i] * W.E[i];
    W.l[i] = lo; W.u[i] = hi;
    W.ctype[i] = constraint_type(lo, hi);
  }
  __syncthreads();
  Rho rv(rho);
  clk.lap(OCP_B200_PHASE_SCALE);
  tri_assemble(P, W, rv, sigma);
  clk.lap(OCP_B200_PHASE_KKT_ASSEMBLE);
  factor_dispatch<kPlace>(P, W);
  clk.lap(OCP_B200_PHASE_FACTOR);

  const PatternOps I{P};
  const int interval = rho_interval(S);
  int status = OCP_B200_QP_UNSOLVED, iter = 0, solves = 0, rho_updates = 0, checks = 0, n_trace = 0;
  double prim_res = 0.0, dual_res = 0.0;
  bool done = false;

  for (iter = 1; iter <= S.admm_max_iter && !done; ++iter) {
    // ---- right-hand side of the reduced KKT system: sigma x - q + A'(rho z - y) --------------
    for (int j = tid; j < n; j += T) {
      double s = sigma * W.x[j] - W.q[j];
      W.b[j] = s + col_dot_A(P, W.Aval, W.w, j);
    }
    __syncthreads();
    clk.lap(OCP_B200_PHASE_RHS);
    solve_dispatch<kPlace>(P, W);   // b <- x~
    ++solves;
    clk.lap(OCP_B200_PHASE_SOLVE);

    // ---- x, z, y updates with relaxation and projection (update_x / update_z / update_y) ----
    const IterFlags F(S, interval, iter);
    const bool want_info = F.want_info();
    for_rows_A(P, W.Aval, W.b, [&](int i, double zt) {
      const signed char ct = W.ctype[i];
      const double rh = rv.of(ct);
      const double zr = relax * zt + (1.0 - relax) * W.z[i];
      const double zn = fmin(fmax(zr + rv.inv(ct) * W.y[i], W.l[i]), W.u[i]);
      const double dy = rh * (zr - zn);
      const double yn = W.y[i] + dy;
      W.y[i] = yn;
      W.z[i] = zn;
      W.w[i] = rh * zn - yn;
      if (want_info) W.dy[i] = dy;
    });
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
      for (int i = tid; i < m; i += T) W.w[i] = rv.of(W.ctype[i]) * W.z[i] - W.y[i];
      tri_assemble(P, W, rv, sigma);
      factor_dispatch<kPlace>(P, W);
    }
    clk.lap(OCP_B200_PHASE_CHECK);
  }
  if (!done) status = OCP_B200_QP_MAX_ITER_REACHED;
  if (A.trace && inst == 0 && tid == 0 && A.n_trace) *A.n_trace = n_trace;
  out = QpResult{status, done ? iter - 1 : S.admm_max_iter, solves, rho_updates, checks, prim_res, dual_res, rho};
  store_solution(qp_vectors(W, n, m), status, cinv);
}

// persistent kernel: CTAs pull instances from A.counter
template <int kPlace, int kThreads, int kBlocksPerSm>
__global__ void __launch_bounds__(kThreads, kBlocksPerSm)
admm_direct_kernel(const PatternDev P, const ocp_b200_settings S, const SolveArgs A, const uint32_t smem_mask) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red_buf[2 * (kThreads / 32) * kRedWidth];
  __shared__ int s_inst;
  __shared__ unsigned long long ring_bar[2 * kMaxRing];
  __shared__ unsigned ring_phase[2];
  Work W;
  carve<kPlace>(W, P, smem_mask, reinterpret_cast<double*>(smem_raw),
                A.slab + size_t(blockIdx.x) * A.slab_doubles);
  W.ring_bar = ring_bar; W.ring_phase = ring_phase;
  // PLACE_BIG: the staging area is split between the two chains of the twisted sweeps; PLACE_MIXED
  // (generic block code, one chain): the whole area is one ring, provided it is in shared memory and
  // the factor is not
  W.ring_slots = (kPlace == PLACE_BIG && P.stage_slots >= 6) ? min(P.stage_slots / 2, kMaxRing) : 0;
  if (kPlace == PLACE_MIXED && !exact_block_code(P) && (smem_mask >> AR_STAGE & 1u) && (smem_mask >> AR_B & 1u) &&
      !(smem_mask >> AR_LSUB & 1u) && !(smem_mask >> AR_DINV & 1u))
    W.ring_slots = min((P.stage_slots > 0 ? P.stage_slots : 4) + ((smem_mask >> AR_SCRATCH & 1u) ? 2 : 0), kMaxRing);
  if ((kPlace == PLACE_BIG || kPlace == PLACE_MIXED) && threadIdx.x == 0) {
    for (int i = 0; i < 2 * kMaxRing; ++i)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(ring_bar + i))));
    ring_phase[0] = 0u; ring_phase[1] = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  PatternDev PL = P;
  if (kPlace != PLACE_MIXED || (smem_mask >> AR_IDX & 1u)) {
    // index structures move into shared memory once per CTA (same offsets as the global arena)
    for (int k = threadIdx.x; k < P.idx_entries; k += blockDim.x) W.idx[k] = P.idx_base[k];
    auto move = [&](const idx_t*& ptr) { ptr = W.idx + (ptr - P.idx_base); };
    move(PL.a_colptr); move(PL.a_rowidx); move(PL.a_rowptr); move(PL.a_colidx); move(PL.a_perm);
    move(PL.p_colptr); move(PL.p_rowidx); move(PL.rows_long); move(PL.rows_short);
    __syncthreads();
  }
  Reducer R{red_buf, 0, (kThreads / 32) * kRedWidth};
  for (int inst; (inst = next_instance(A, s_inst)) < A.B;) {
    QpResult res;
    solve_instance<kPlace>(PL, S, A, W, R, inst, res);
    write_outputs(P, A, W.x, W.y, R, inst, res);
  }
  if (kCanaryDoubles > 0) {
    __syncthreads();
    Work W2;
    carve<kPlace>(W2, P, smem_mask, reinterpret_cast<double*>(smem_raw),
                  A.slab + size_t(blockIdx.x) * A.slab_doubles, true);
  }
}

}  // namespace direct
}  // namespace ocpb200
