// admm_common.cuh -- pieces shared by the batched ADMM QP kernels for sm_100a
// (admm_direct_kernel.cuh: bordered block-tridiagonal LDL' of the reduced KKT matrix;
//  admm_compact_kernel.cuh: the same solve with the per-instance state packed for four CTAs per SM;
//  admm_pcg_kernel.cuh: preconditioned CG on the same matrix for patterns without that structure),
// among them the whole OSQP decision layer (update_info, check_termination, adapt_rho, store_solution).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "ocp_b200.h"

namespace ocpb200 {

constexpr double kInfty = 1e30, kMinScaling = 1e-4, kMaxScaling = 1e4;
constexpr double kRhoMin = 1e-6, kRhoMax = 1e6, kRhoTol = 1e-4, kRhoEqOverIneq = 1e3;
constexpr double kDivisionTol = 1e-30;
constexpr int kRedWidth = 16;          // max values per block reduction
constexpr int kMaxWarps = 32;

typedef uint16_t idx_t;

// -DOCP_B200_CANARY: every per-instance array (shared memory and slab) is followed by two guard doubles that the
// kernels fill when they carve their state and verify when they leave; an overwritten guard is reported with
// printf ("OCP_B200 CANARY ...").  compute-sanitizer is closed on the GPU pool this was developed on: this is the
// bounds check of our own (tools/sanitize_cases.py runs every placement with it, profiles/r2_canary.txt).
#ifdef OCP_B200_CANARY
constexpr int kCanaryDoubles = 2;
#else
constexpr int kCanaryDoubles = 0;
#endif
__device__ __forceinline__ double canary_value(int id) { return __longlong_as_double(0x7ff4dead00000000LL + id); }

// K-assembly program (direct kernel): one entry per structurally non-zero element of the bordered
// block-tridiagonal K = P + sigma I + A' diag(rho) A that has to be computed, with the products
// sum_r rho_r A_ri A_rj encoded as RUNS of consecutive positions in columns i and j of A whose rows
// coincide one-to-one AND are consecutive rows row0, row0 + 1, ... (host-side merge of the two sorted
// columns, done once per pattern), so that the constraint type of every product needs no index lookup.
struct KRun { uint16_t ka, kc, len, row0; };
struct KEntry {
  uint32_t dest0, dest1;   // (array << 30) | offset; array 0 = Dinv, 1 = Lsub, 2 = Lp, 3 = Dp; dest1 = mirror or 0xffffffff
  int32_t ppos;            // position of P_ij in the symmetrised P values, or -1
  uint32_t run_begin;      // first run in the run array
  uint16_t nruns, diag;    // diag != 0: i == j (sigma is added)
  uint32_t pad;
};

// Index structures of one sparsity pattern (device pointers, shared by every instance)
struct PatternDev {
  int n, m, nnz_a, nnz_p, nnz_h;
  int nblk, minv_doubles, max_bs;
  int n_long, n_short;
  // bordered block-tridiagonal structure of K = P + sigma I + A' diag(rho) A (direct kernel):
  // columns [0, tri_np) form the border (the reference parameters p), then tri_nb diagonal
  // blocks of tri_bs columns each; block rows are stored with an even pitch tri_ld >= tri_bs + 1
  int tri_ok, tri_np, tri_bs, tri_nb, tri_ld;
  int stage_slots;         // block staging buffers per CTA when the factor is slab-resident (4, or 8 = a ring of 4 per chain)
  int kprog_entries;       // K-assembly program (null / 0: assemble by merging columns on the device)
  const KEntry* kprog;
  const KRun* kruns;
  int idx_entries;         // length of the idx_t arena (every array padded to 8 entries)
  const idx_t* idx_base;   // start of the arena
  const idx_t* a_colptr;   // n+1
  const idx_t* a_rowidx;   // nnz_a
  const idx_t* a_rowptr;   // m+1
  const idx_t* a_colidx;   // nnz_a, CSR order
  const idx_t* a_perm;     // nnz_a, CSR position -> CSC position
  const idx_t* p_colptr;   // n+1   (symmetrised full pattern of the upper triangle of H)
  const idx_t* p_rowidx;   // nnz_p
  const int* p_src;        // nnz_p, index into the caller's H values (upper-triangle twin)
  const idx_t* blk_ptr;    // nblk+1
  const idx_t* blk_of_col; // n
  const int* minv_off;     // nblk
  const idx_t* rows_long;  // rows handled by 4 lanes each
  const idx_t* rows_short; // rows handled by one thread each
};

struct SolveArgs {
  int B;
  // QP data, one row per instance
  const double* h_vals; int ld_h;
  const double* q; int ld_n;
  const double* a_vals; int ld_a;
  const double* l; const double* u; int ld_m;
  // outputs
  double* sol_x;      // B*n   unscaled primal solution (may be null)
  double* sol_y;      // B*m   unscaled dual solution (may be null)
  double* info;       // B*OCP_B200_NINFO (may be null)
  // SQP update: x_iter[b*N + i] += alpha * sol[np + i]; stats accumulated (may be null)
  double* x_iter; int np; int N; double sqp_alpha;
  double* stats; int first_step;
  // trace of instance 0 (may be null)
  double* trace; int max_trace; int* n_trace;
  // optional phase cycle counters of CTA 0 (OCP_B200_NPHASE long longs, may be null)
  long long* phase;
  // scheduling + streaming workspace
  int* counter;
  double* slab; size_t slab_doubles;
};

// ---------------------------------------------------------------------------------------
// block reductions: warp shuffles, then one shared-memory exchange; every thread returns
// with the same result.  Two alternating exchange buffers make one barrier per call enough.
// ---------------------------------------------------------------------------------------
struct Reducer {
  double* buf;   // 2 * half doubles of shared memory, half >= (warps per CTA) * kRedWidth
  int parity;
  int half;
};

template <int NV, bool kMax>
__device__ __forceinline__ void block_reduce(double (&v)[NV], Reducer& R) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    double a = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double b = __shfl_xor_sync(0xffffffffu, a, o);
      a = kMax ? fmax(a, b) : a + b;
    }
    v[k] = a;
  }
  double* buf = R.buf + R.parity * R.half;
  R.parity ^= 1;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) buf[warp * NV + k] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    double a = buf[k];
    for (int w = 1; w < nw; ++w) a = kMax ? fmax(a, buf[w * NV + k]) : a + buf[w * NV + k];
    v[k] = a;
  }
}

__device__ __forceinline__ double limit_scaling(double v) {
  v = v < kMinScaling ? 1.0 : v;
  return v > kMaxScaling ? kMaxScaling : v;
}

// ---------------------------------------------------------------------------------------
// sparse kernels over one instance.  A rows go through the CSR view (values fetched
// through the CSR->CSC permutation), A and P columns through the CSC arrays.
// ---------------------------------------------------------------------------------------
template <typename F>
__device__ __forceinline__ void for_rows_A(const PatternDev& P, const double* __restrict__ Aval,
                                           const double* __restrict__ src, F f) {
  const int tid = threadIdx.x, T = blockDim.x;
  // long rows: 4 lanes per row
  for (int base = 0; base < P.n_long; base += (T >> 2)) {
    const int idx = base + (tid >> 2);
    const bool valid = idx < P.n_long;
    double s = 0.0;
    int row = 0;
    if (valid) {
      row = P.rows_long[idx];
      const int e = P.a_rowptr[row + 1];
#pragma unroll 4
      for (int k = P.a_rowptr[row] + (tid & 3); k < e; k += 4) s += Aval[P.a_perm[k]] * src[P.a_colidx[k]];
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (valid && (tid & 3) == 0) f(row, s);
  }
  for (int idx = tid; idx < P.n_short; idx += T) {
    const int row = P.rows_short[idx];
    double s = 0.0;
    const int e = P.a_rowptr[row + 1];
#pragma unroll 4
    for (int k = P.a_rowptr[row]; k < e; ++k) s += Aval[P.a_perm[k]] * src[P.a_colidx[k]];
    f(row, s);
  }
}

__device__ __forceinline__ double col_dot_A(const PatternDev& P, const double* __restrict__ Aval,
                                            const double* __restrict__ v, int j) {
  double s = 0.0;
  const int e = P.a_colptr[j + 1];
#pragma unroll 4
  for (int k = P.a_colptr[j]; k < e; ++k) s += Aval[k] * v[P.a_rowidx[k]];
  return s;
}
__device__ __forceinline__ double col_dot_P(const PatternDev& P, const double* __restrict__ Pval,
                                            const double* __restrict__ v, int j) {
  double s = 0.0;
  const int e = P.p_colptr[j + 1];
#pragma unroll 4
  for (int k = P.p_colptr[j]; k < e; ++k) s += Pval[k] * v[P.p_rowidx[k]];
  return s;
}

// The sparse products of the OSQP layer below over the CSC / CSR arrays of PatternDev (direct and PCG kernels;
// the compact kernel has its own over the stage-periodic templates).
struct PatternOps {
  const PatternDev& P;
  template <typename F>
  __device__ __forceinline__ void for_rows_A(const double* Aval, const double* src, F f) const { ocpb200::for_rows_A(P, Aval, src, f); }
  __device__ __forceinline__ double col_dot_A(const double* Aval, const double* v, int j) const { return ocpb200::col_dot_A(P, Aval, v, j); }
  __device__ __forceinline__ double col_dot_P(const double* Pval, const double* v, int j) const { return ocpb200::col_dot_P(P, Pval, v, j); }
};

// cycle accounting of CTA 0 (diagnostics; see ocp_b200_get_phase_cycles)
struct PhaseClock {
  long long* out; long long t0;
  __device__ PhaseClock(long long* o) : out((blockIdx.x == 0 && threadIdx.x == 0) ? o : nullptr), t0(0) { if (out) t0 = clock64(); }
  __device__ __forceinline__ void lap(int phase) {
    if (out) { const long long t = clock64(); out[phase] += t - t0; t0 = t; }
  }
};


// The finer split of the solve / factor phases costs a predicated branch per lap in every thread;
// it is compiled in only with -DOCP_B200_FINE_PHASES (tools/phase_profile.py documents the numbers).
#ifdef OCP_B200_FINE_PHASES
#define OCP_B200_FINE_CLOCK(name, ptr) PhaseClock name(ptr)
#define OCP_B200_FINE_LAP(name, phase) name.lap(phase)
#else
#define OCP_B200_FINE_CLOCK(name, ptr)
#define OCP_B200_FINE_LAP(name, phase)
#endif

struct QpResult {
  int status, iters, pcg_iters, rho_updates, checks;
  double prim_res, dual_res, rho;
};

// per-instance outputs after a QP: solution, SQP update x += alpha * d[np:], info / stats.
// xs / ys: unscaled primal / dual solution of the instance (any address space).
__device__ inline void write_outputs(const PatternDev& P, const SolveArgs& A, const double* xs, const double* ys,
                                      Reducer& R, int inst, const QpResult& res) {
  const bool solved_setup = res.status != OCP_B200_QP_UNSOLVED || res.iters > 0;
  if (A.sol_x)
    for (int j = threadIdx.x; j < P.n; j += blockDim.x) A.sol_x[size_t(inst) * P.n + j] = solved_setup ? xs[j] : 0.0;
  if (A.sol_y)
    for (int i = threadIdx.x; i < P.m; i += blockDim.x) A.sol_y[size_t(inst) * P.m + i] = solved_setup ? ys[i] : 0.0;
  double nrm[1] = {0.0};
  if (A.x_iter) {
    double* xi = A.x_iter + size_t(inst) * A.N;
    for (int i = threadIdx.x; i < A.N; i += blockDim.x) {
      const double dx = solved_setup ? A.sqp_alpha * xs[A.np + i] : 0.0;
      xi[i] += dx;
      nrm[0] += dx * dx;
    }
    block_reduce<1, false>(nrm, R);
  }
  if (threadIdx.x == 0) {
    if (A.info) {
      double* f = A.info + size_t(inst) * OCP_B200_NINFO;
      f[OCP_B200_INFO_STATUS] = res.status; f[OCP_B200_INFO_ITERS] = res.iters;
      f[OCP_B200_INFO_PCG_ITERS] = res.pcg_iters; f[OCP_B200_INFO_PRIM_RES] = res.prim_res;
      f[OCP_B200_INFO_DUAL_RES] = res.dual_res; f[OCP_B200_INFO_RHO] = res.rho;
      f[OCP_B200_INFO_RHO_UPDATES] = res.rho_updates; f[OCP_B200_INFO_CHECKS] = res.checks;
    }
    if (A.stats) {
      double* s = A.stats + size_t(inst) * OCP_B200_NSTATS;
      if (A.first_step) for (int k = 0; k < OCP_B200_NSTATS; ++k) s[k] = 0.0;
      s[OCP_B200_STAT_QP_STATUS] = res.status;
      s[OCP_B200_STAT_SQP_STEPS] += 1.0;
      s[OCP_B200_STAT_ADMM_ITERS] += res.iters;
      s[OCP_B200_STAT_PCG_ITERS] += res.pcg_iters;
      s[OCP_B200_STAT_PRIM_RES] = res.prim_res;
      s[OCP_B200_STAT_DUAL_RES] = res.dual_res;
      s[OCP_B200_STAT_RHO_UPDATES] += res.rho_updates;
      s[OCP_B200_STAT_LAST_ADMM] = res.iters;
      s[OCP_B200_STAT_LAST_RHO] = res.rho;
      s[OCP_B200_STAT_CHECKS] += res.checks;
      s[OCP_B200_STAT_STEP_NORM] = sqrt(nrm[0]);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------
// The OSQP decision layer of the three kernels: residuals, termination and infeasibility
// certificates, rho adaptation, trace and solution store.  The sparse products go through
// Ops (PatternOps, or compact::CompactOps), which supplies col_dot_A, col_dot_P and
// for_rows_A; each kernel keeps its own row product and reduction order.
// ---------------------------------------------------------------------------------------

// persistent kernels: the CTA pulls its next instance from A.counter (done at A.B);
// s_inst: one int of shared memory
__device__ __forceinline__ int next_instance(const SolveArgs& A, int& s_inst) {
  if (threadIdx.x == 0) s_inst = atomicAdd(A.counter, 1);
  __syncthreads();
  const int inst = s_inst;
  __syncthreads();
  return inst;
}

// set_rho_vec: -1 free (both bounds infinite), 1 equality, 0 inequality, from the scaled bounds
__device__ __forceinline__ signed char constraint_type(double lo, double hi) {
  if (lo < -kInfty * kMinScaling && hi > kInfty * kMinScaling) return -1;
  return hi - lo < kRhoTol ? 1 : 0;
}

// OSQP without wall-clock profiling: 4 x check_termination, or ADAPTIVE_RHO_FIXED = 100 iterations when checks are off
__device__ __forceinline__ int rho_interval(const ocp_b200_settings& S) {
  return S.adaptive_rho_interval > 0 ? S.adaptive_rho_interval : (S.check_termination > 0 ? 4 * S.check_termination : 100);
}

// what ADMM iteration iter (1-based) does after its update: residuals are needed for any of the three
struct IterFlags {
  bool can_check, last_iter, rho_time;
  __device__ __forceinline__ IterFlags(const ocp_b200_settings& S, int interval, int iter)
      : can_check(S.check_termination > 0 && (iter % S.check_termination == 0)),
        last_iter(iter == S.admm_max_iter),
        rho_time(S.adaptive_rho && interval > 0 && (iter % interval == 0)) {}
  __device__ __forceinline__ bool want_info() const { return can_check || rho_time || last_iter; }
};

// The per-instance vectors of the scaled problem the decision layer reads, wherever the kernel keeps them
// (shared memory or slab).  dx, dy: the last ADMM step; is_primal_infeasible projects dy in place,
// store_solution unscales x and y in place.
struct QpVec {
  int n, m;
  const double *Aval, *Pval, *q, *l, *u, *D, *E, *z;
  double *x, *y, *dx, *dy;
};
// (built where it is used: pointers held across the iteration loop cost registers in every phase, DESIGN.md 5.5)
template <class Work>
__device__ __forceinline__ QpVec qp_vectors(const Work& W, int n, int m) {
  return QpVec{n, m, W.Aval, W.Pval, W.q, W.l, W.u, W.D, W.E, W.z, W.x, W.y, W.dx, W.dy};
}

// update_info: the inf-norms behind the residuals and their tolerances, unscaled (U) and scaled (S).
// Kept as one array so that one block reduction of kRedWidth values serves them all.
enum InfoSlot {
  kPrimU, kAxU, kZU,          // E^-1 (Ax - z), E^-1 Ax, E^-1 z
  kPrimS, kAxS, kZS,          //      Ax - z,        Ax,       z
  kDualU, kQU, kPxU, kAtyU,   // D^-1 (q + Px + A'y), D^-1 q, D^-1 Px, D^-1 A'y  (times 1/c when used)
  kDualS, kQS, kPxS, kAtyS,   //      q + Px + A'y,        q,      Px,      A'y
  kNumInfo
};
static_assert(kNumInfo <= kRedWidth, "the residual norms are reduced in one call");

template <class Ops>
__device__ __forceinline__ void update_info(const Ops& I, const QpVec& V, Reducer& R, double (&mx)[kRedWidth]) {
#pragma unroll
  for (int k = 0; k < kRedWidth; ++k) mx[k] = 0.0;
  I.for_rows_A(V.Aval, V.x, [&](int i, double ax) {
    const double einv = 1.0 / V.E[i];
    const double zi = V.z[i];
    const double rp = ax - zi;
    mx[kPrimU] = fmax(mx[kPrimU], fabs(einv * rp));
    mx[kAxU] = fmax(mx[kAxU], fabs(einv * ax));
    mx[kZU] = fmax(mx[kZU], fabs(einv * zi));
    mx[kPrimS] = fmax(mx[kPrimS], fabs(rp));
    mx[kAxS] = fmax(mx[kAxS], fabs(ax));
    mx[kZS] = fmax(mx[kZS], fabs(zi));
  });
  for (int j = threadIdx.x; j < V.n; j += blockDim.x) {
    const double dinv = 1.0 / V.D[j];
    const double qj = V.q[j];
    const double px = I.col_dot_P(V.Pval, V.x, j);
    const double aty = I.col_dot_A(V.Aval, V.y, j);
    const double rd = qj + px + aty;
    mx[kDualU] = fmax(mx[kDualU], fabs(dinv * rd));
    mx[kQU] = fmax(mx[kQU], fabs(dinv * qj));
    mx[kPxU] = fmax(mx[kPxU], fabs(dinv * px));
    mx[kAtyU] = fmax(mx[kAtyU], fabs(dinv * aty));
    mx[kDualS] = fmax(mx[kDualS], fabs(rd));
    mx[kQS] = fmax(mx[kQS], fabs(qj));
    mx[kPxS] = fmax(mx[kPxS], fabs(px));
    mx[kAtyS] = fmax(mx[kAtyS], fabs(aty));
  }
  block_reduce<kRedWidth, true>(mx, R);
}

// residuals of the unscaled problem (c: cost scaling of the Ruiz equilibration, cinv = 1 / c)
__device__ __forceinline__ double prim_residual(const double (&mx)[kRedWidth]) { return mx[kPrimU]; }
__device__ __forceinline__ double dual_residual(const double (&mx)[kRedWidth], double cinv) { return cinv * mx[kDualU]; }

// after the last iteration without a decision: the test with 10x tolerances
__device__ __forceinline__ int approximate_status(const ocp_b200_settings& S, const double (&mx)[kRedWidth], double cinv) {
  const double ep = 10.0 * S.eps_abs + 10.0 * S.eps_rel * fmax(mx[kZU], mx[kAxU]);
  const double ed = 10.0 * S.eps_abs + 10.0 * S.eps_rel * cinv * fmax(mx[kQU], fmax(mx[kAtyU], mx[kPxU]));
  return prim_residual(mx) < ep && dual_residual(mx, cinv) < ed
             ? OCP_B200_QP_SOLVED_INACCURATE : OCP_B200_QP_MAX_ITER_REACHED;
}

// check_termination: SOLVED, PRIMAL_INFEASIBLE or DUAL_INFEASIBLE, or -1 to continue
template <class Ops>
__device__ __forceinline__ int check_termination(const Ops& I, const QpVec& V, const ocp_b200_settings& S, Reducer& R,
                                                 const double (&mx)[kRedWidth], double c, double cinv) {
  const int tid = threadIdx.x, T = blockDim.x, n = V.n, m = V.m;
  const double eps_prim = S.eps_abs + S.eps_rel * fmax(mx[kZU], mx[kAxU]);
  const double eps_dual = S.eps_abs + S.eps_rel * cinv * fmax(mx[kQU], fmax(mx[kAtyU], mx[kPxU]));
  const bool prim_ok = prim_residual(mx) < eps_prim, dual_ok = dual_residual(mx, cinv) < eps_dual;
  bool prim_inf = false, dual_inf = false;
  if (!prim_ok) {
    // is_primal_infeasible: dy projected on the polar of the recession cone of [l, u]
    double a2[1] = {0.0};
    for (int i = tid; i < m; i += T) {
      double dy = V.dy[i];
      const double lo = V.l[i], hi = V.u[i];
      if (hi > kInfty * kMinScaling) {
        if (lo < -kInfty * kMinScaling) dy = 0.0; else dy = fmin(dy, 0.0);
      } else if (lo < -kInfty * kMinScaling) {
        dy = fmax(dy, 0.0);
      }
      V.dy[i] = dy;
      a2[0] = fmax(a2[0], fabs(V.E[i] * dy));
    }
    // (the barrier of this reduction also orders the dy writes before the A' dy gather below)
    block_reduce<1, true>(a2, R);
    const double norm_dy = a2[0];
    if (norm_dy > kDivisionTol) {
      double lhs[1] = {0.0};
      for (int i = tid; i < m; i += T) lhs[0] += V.u[i] * fmax(V.dy[i], 0.0) + V.l[i] * fmin(V.dy[i], 0.0);
      block_reduce<1, false>(lhs, R);
      if (lhs[0] < -S.eps_prim_inf * norm_dy) {
        double na[1] = {0.0};
        for (int j = tid; j < n; j += T) na[0] = fmax(na[0], fabs(I.col_dot_A(V.Aval, V.dy, j) / V.D[j]));
        block_reduce<1, true>(na, R);
        prim_inf = na[0] < S.eps_prim_inf * norm_dy;
      }
    }
  }
  if (!dual_ok) {
    // is_dual_infeasible
    double a2[1] = {0.0};
    for (int j = tid; j < n; j += T) a2[0] = fmax(a2[0], fabs(V.D[j] * V.dx[j]));
    block_reduce<1, true>(a2, R);
    const double norm_dx = a2[0];
    if (norm_dx > kDivisionTol) {
      double qdx[1] = {0.0};
      for (int j = tid; j < n; j += T) qdx[0] += V.q[j] * V.dx[j];
      block_reduce<1, false>(qdx, R);
      if (qdx[0] < -c * S.eps_dual_inf * norm_dx) {
        double np_[1] = {0.0};
        for (int j = tid; j < n; j += T) np_[0] = fmax(np_[0], fabs(I.col_dot_P(V.Pval, V.dx, j) / V.D[j]));
        block_reduce<1, true>(np_, R);
        if (np_[0] < c * S.eps_dual_inf * norm_dx) {
          double viol[1] = {0.0};
          I.for_rows_A(V.Aval, V.dx, [&](int i, double adx) {
            const double a = adx / V.E[i];
            if ((V.u[i] < kInfty * kMinScaling && a > S.eps_dual_inf * norm_dx) ||
                (V.l[i] > -kInfty * kMinScaling && a < -S.eps_dual_inf * norm_dx)) viol[0] = 1.0;
          });
          block_reduce<1, true>(viol, R);
          dual_inf = viol[0] == 0.0;
        }
      }
    }
  }
  if (prim_ok && dual_ok) return OCP_B200_QP_SOLVED;
  if (prim_inf) return OCP_B200_QP_PRIMAL_INFEASIBLE;
  return dual_inf ? OCP_B200_QP_DUAL_INFEASIBLE : -1;
}

// adapt_rho: estimate from the SCALED residuals; true, with rho set to the estimate, when it moved by more
// than adaptive_rho_tolerance (the caller then rebuilds its linear system)
__device__ __forceinline__ bool adapt_rho(const ocp_b200_settings& S, const double (&mx)[kRedWidth], double& rho) {
  const double pr = mx[kPrimS] / (fmax(mx[kZS], mx[kAxS]) + 1e-10);
  const double dr = mx[kDualS] / (fmax(mx[kQS], fmax(mx[kAtyS], mx[kPxS])) + 1e-10);
  double est = rho * sqrt(pr / (dr + 1e-10));
  est = fmin(fmax(est, kRhoMin), kRhoMax);
  if (!(est > rho * S.adaptive_rho_tolerance || est < rho / S.adaptive_rho_tolerance)) return false;
  rho = est;
  return true;
}

// one row of the check trace of instance 0: iteration, residuals, rho, linear solves so far, status of the check
__device__ __forceinline__ void record_trace(const SolveArgs& A, int inst, int& n_trace, int iter, double prim_res,
                                             double dual_res, double rho, int solves, int st) {
  if (!(A.trace && inst == 0 && n_trace < A.max_trace)) return;
  if (threadIdx.x == 0) {
    double* tr = A.trace + size_t(n_trace) * OCP_B200_TRACE_WIDTH;
    tr[0] = iter; tr[1] = prim_res; tr[2] = dual_res; tr[3] = rho; tr[4] = solves;
    tr[5] = st < 0 ? OCP_B200_QP_UNSOLVED : st;
  }
  ++n_trace;
}

// store_solution: unscale in place (x <- D x, y <- E y / c), or NaN for a certificate
__device__ __forceinline__ void store_solution(const QpVec& V, int status, double cinv) {
  const bool has_sol = status != OCP_B200_QP_PRIMAL_INFEASIBLE && status != OCP_B200_QP_DUAL_INFEASIBLE;
  const double nanv = __longlong_as_double(0x7ff8000000000000LL);
  for (int j = threadIdx.x; j < V.n; j += blockDim.x) V.x[j] = has_sol ? V.D[j] * V.x[j] : nanv;
  for (int i = threadIdx.x; i < V.m; i += blockDim.x) V.y[i] = has_sol ? cinv * V.E[i] * V.y[i] : nanv;
  __syncthreads();
}

}  // namespace ocpb200
