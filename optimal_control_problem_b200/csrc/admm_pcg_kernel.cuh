// admm_kernel.cuh -- batched ADMM QP solver for sm_100a, one CTA per instance.
//
// Replaces, for B independent QPs that share one sparsity pattern, what the reference does
// per SQP step through OsqpEigen/OSQP (src/sqp_solver/CuCaQP.cpp:271-288, 183-224):
//   osqp_setup : bound clamping, Ruiz equilibration x10 with cost normalisation, rho vector,
//                linear-system set-up, cold start
//   osqp_solve : ADMM iterations, residual / termination / infeasibility checks every 25
//                iterations, adaptive rho, unscaling of the solution
// and, after the QP, the SQP update x += alpha * d[np:] (SQPOptimizationSolver.cpp:171-177).
//
// Linear system: OSQP's indirect formulation (its cuda backend): the reduced KKT system
//   (P + sigma I + A' diag(rho) A) x~ = sigma x - q + A'(rho z - y),   z~ = A x~
// solved by preconditioned CG, warm-started from the previous x~, stopped on the relative
// residual.  With a tight tolerance the iterates coincide with those of the direct LDL'
// solve the reference's CPU build uses (oracle/osqp_restate.hpp), which is what the parity
// tests check.
//
// Layout: a persistent CTA takes instances from an atomic counter.  All per-instance state
// (matrix values, 19 vectors, preconditioner blocks) lives in shared memory when it fits
// ("resident", the quadrotor shape), otherwise in a per-CTA slab of global memory that stays
// L2-resident ("streaming").  Index structures are shared by the whole batch.  No host
// round trip happens inside a QP solve: termination, rho updates and preconditioner
// rebuilds are decided on the device.
#pragma once

#include "admm_common.cuh"

namespace ocpb200 {
namespace pcg {

// Where the per-instance state lives (shared memory or a global slab)
struct Work {
  double *Aval, *Pval;
  double *x, *xt, *q, *r, *d, *Kd, *zc, *D, *dx;          // n
  double *z, *zt, *y, *l, *u, *E, *w, *t, *dy, *rho;      // m
  double *Minv;
  signed char* ctype;                                      // m
};

__host__ __device__ inline size_t work_doubles(const PatternDev& P) {
  return size_t(P.nnz_a) + P.nnz_p + 9 * size_t(P.n) + 10 * size_t(P.m) + P.minv_doubles + (P.m + 7) / 8;
}
// index entries the resident kernel stages in shared memory behind its state: the arrays of the stage(...) list in
// admm_solve_kernel, each padded to 8 entries -- the two must list the same arrays
__host__ __device__ inline size_t staged_idx_entries(const PatternDev& P) {
  auto pad8 = [](size_t v) { return (v + 7) & ~size_t(7); };
  return 2 * pad8(P.n + 1) + 3 * pad8(P.nnz_a) + pad8(P.m + 1) + pad8(P.nnz_p) + pad8(P.nblk + 1) + pad8(P.n) +
         pad8(P.n_long) + pad8(P.n_short);
}

__device__ inline void carve(Work& W, double* base, const PatternDev& P) {
  double* p = base;
  W.Aval = p; p += P.nnz_a;
  W.Pval = p; p += P.nnz_p;
  double** nv[9] = {&W.x, &W.xt, &W.q, &W.r, &W.d, &W.Kd, &W.zc, &W.D, &W.dx};
  for (int k = 0; k < 9; ++k) { *nv[k] = p; p += P.n; }
  double** mv[10] = {&W.z, &W.zt, &W.y, &W.l, &W.u, &W.E, &W.w, &W.t, &W.dy, &W.rho};
  for (int k = 0; k < 10; ++k) { *mv[k] = p; p += P.m; }
  W.Minv = p; p += P.minv_doubles;
  W.ctype = reinterpret_cast<signed char*>(p);
}

// ---------------------------------------------------------------------------------------
// preconditioner: inverse of the diagonal blocks of K = P + sigma I + A' diag(rho) A
// (block size 1 for OCP_B200_PRECOND_DIAGONAL)
// ---------------------------------------------------------------------------------------
__device__ inline void build_preconditioner(const PatternDev& P, const Work& W, double sigma, int precond) {
  const int tid = threadIdx.x, T = blockDim.x;
  if (precond == OCP_B200_PRECOND_DIAGONAL) {
    for (int j = tid; j < P.n; j += T) {
      double s = sigma;
      for (int k = P.p_colptr[j]; k < P.p_colptr[j + 1]; ++k)
        if (P.p_rowidx[k] == j) s += W.Pval[k];
      for (int k = P.a_colptr[j]; k < P.a_colptr[j + 1]; ++k) s += W.rho[P.a_rowidx[k]] * W.Aval[k] * W.Aval[k];
      W.Minv[j] = 1.0 / s;
    }
    __syncthreads();
    return;
  }
  // dense diagonal blocks: entry (a, c), a <= c, by a sorted merge of the two A columns
  for (int b = 0; b < P.nblk; ++b) {
    const int j0 = P.blk_ptr[b], bs = P.blk_ptr[b + 1] - j0;
    double* M = W.Minv + P.minv_off[b];
    for (int pidx = tid; pidx < bs * bs; pidx += T) {
      const int a = pidx / bs, c = pidx - a * bs;
      if (a > c) continue;
      const int ja = j0 + a, jc = j0 + c;
      double s = (a == c) ? sigma : 0.0;
      for (int k = P.p_colptr[jc]; k < P.p_colptr[jc + 1]; ++k)
        if (P.p_rowidx[k] == ja) s += W.Pval[k];
      int ka = P.a_colptr[ja], kc = P.a_colptr[jc];
      const int ea = P.a_colptr[ja + 1], ec = P.a_colptr[jc + 1];
      while (ka < ea && kc < ec) {
        const int ra = P.a_rowidx[ka], rc = P.a_rowidx[kc];
        if (ra == rc) { s += W.rho[ra] * W.Aval[ka] * W.Aval[kc]; ++ka; ++kc; }
        else if (ra < rc) ++ka;
        else ++kc;
      }
      M[a * bs + c] = s;
      M[c * bs + a] = s;
    }
  }
  __syncthreads();
  // in-place Gauss-Jordan inverse (SPD: no pivoting), one warp per block
  const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
  for (int b = warp; b < P.nblk; b += nw) {
    const int bs = P.blk_ptr[b + 1] - P.blk_ptr[b];
    double* M = W.Minv + P.minv_off[b];
    for (int k = 0; k < bs; ++k) {
      const double ipiv = 1.0 / M[k * bs + k];
      __syncwarp();
      for (int c = lane; c < bs; c += 32) M[k * bs + c] = (c == k) ? ipiv : M[k * bs + c] * ipiv;
      __syncwarp();
      for (int idx = lane; idx < bs * bs; idx += 32) {
        const int r = idx / bs, c = idx - r * bs;
        if (r != k && c != k) M[idx] -= M[r * bs + k] * M[k * bs + c];
      }
      __syncwarp();
      for (int r = lane; r < bs; r += 32)
        if (r != k) M[r * bs + k] = -M[r * bs + k] * ipiv;
      __syncwarp();
    }
  }
  __syncthreads();
}

// zc = M^-1 r for the columns this thread owns (j = tid, tid + T, ...); returns sum r_j zc_j
__device__ __forceinline__ double apply_preconditioner(const PatternDev& P, const Work& W, int precond) {
  const int tid = threadIdx.x, T = blockDim.x;
  double rz = 0.0;
  if (precond == OCP_B200_PRECOND_DIAGONAL) {
    for (int j = tid; j < P.n; j += T) { const double v = W.Minv[j] * W.r[j]; W.zc[j] = v; rz += v * W.r[j]; }
    return rz;
  }
  for (int j = tid; j < P.n; j += T) {
    const int b = P.blk_of_col[j];
    const int j0 = P.blk_ptr[b], bs = P.blk_ptr[b + 1] - j0;
    const double* M = W.Minv + P.minv_off[b] + (j - j0);   // symmetric: column (j - j0), stride bs
    double s = 0.0;
    for (int c = 0; c < bs; ++c) s += M[c * bs] * W.r[j0 + c];
    W.zc[j] = s;
    rz += s * W.r[j];
  }
  return rz;
}

// ---------------------------------------------------------------------------------------
// one QP, solved by the whole CTA
// ---------------------------------------------------------------------------------------
__device__ inline void solve_instance(const PatternDev& P, const ocp_b200_settings& S, const SolveArgs& A,
                                      const Work& W, Reducer& R, int inst, QpResult& out) {
  const int tid = threadIdx.x, T = blockDim.x;
  const int n = P.n, m = P.m;
  const double sigma = S.sigma, relax = S.relax;

  // ---- load (osqp_setup copies its inputs): values, q, bounds clamped to +-1e30 ------------
  {
    const double* hv = A.h_vals + size_t(inst) * A.ld_h;
    const double* av = A.a_vals + size_t(inst) * A.ld_a;
    const double* qv = A.q + size_t(inst) * A.ld_n;
    const double* lv = A.l + size_t(inst) * A.ld_m;
    const double* uv = A.u + size_t(inst) * A.ld_m;
    for (int k = tid; k < P.nnz_a; k += T) W.Aval[k] = av[k];
    for (int k = tid; k < P.nnz_p; k += T) { const int s = P.p_src[k]; W.Pval[k] = s >= 0 ? hv[s] : 0.0; }
    for (int j = tid; j < n; j += T) { W.q[j] = qv[j]; W.D[j] = 1.0; W.x[j] = 0.0; W.xt[j] = 0.0; }
    double bad[1] = {0.0};
    for (int i = tid; i < m; i += T) {
      const double lo = lv[i], hi = uv[i];
      if (lo > hi) bad[0] = 1.0;
      W.l[i] = fmax(lo, -kInfty);
      W.u[i] = fmin(hi, kInfty);
      W.E[i] = 1.0; W.z[i] = 0.0; W.zt[i] = 0.0; W.y[i] = 0.0;
    }
    block_reduce<1, true>(bad, R);
    if (bad[0] > 0.0) {  // osqp_setup rejects l > u; the reference then adds no usable step
      out = QpResult{OCP_B200_QP_UNSOLVED, 0, 0, 0, 0, 0.0, 0.0, S.rho};
      return;
    }
  }

  // ---- Ruiz equilibration (scale_data): D, E, c ----------------------------------------------
  double c = 1.0;
  for (int pass = 0; pass < S.scaling_iters; ++pass) {
    for (int j = tid; j < n; j += T) {
      double dn = 0.0;
      for (int k = P.p_colptr[j]; k < P.p_colptr[j + 1]; ++k) dn = fmax(dn, fabs(W.Pval[k]));
      for (int k = P.a_colptr[j]; k < P.a_colptr[j + 1]; ++k) dn = fmax(dn, fabs(W.Aval[k]));
      W.d[j] = 1.0 / sqrt(limit_scaling(dn));
    }
    for (int i = tid; i < m; i += T) {
      double en = 0.0;
      for (int k = P.a_rowptr[i]; k < P.a_rowptr[i + 1]; ++k) en = fmax(en, fabs(W.Aval[P.a_perm[k]]));
      W.w[i] = 1.0 / sqrt(limit_scaling(en));
    }
    __syncthreads();
    double red[2] = {0.0, 0.0};  // sum of P column norms, max |q|
    for (int j = tid; j < n; j += T) {
      const double dj = W.d[j];
      double cn = 0.0;
      for (int k = P.p_colptr[j]; k < P.p_colptr[j + 1]; ++k) {
        const double v = W.Pval[k] * W.d[P.p_rowidx[k]] * dj;
        W.Pval[k] = v;
        cn = fmax(cn, fabs(v));
      }
      for (int k = P.a_colptr[j]; k < P.a_colptr[j + 1]; ++k) W.Aval[k] *= W.w[P.a_rowidx[k]] * dj;
      const double qj = W.q[j] * dj;
      W.q[j] = qj;
      W.D[j] *= dj;
      red[0] += cn;
      red[1] = fmax(red[1], fabs(qj));
    }
    for (int i = tid; i < m; i += T) W.E[i] *= W.w[i];
    double sum[1] = {red[0]}, mx[1] = {red[1]};
    block_reduce<1, false>(sum, R);
    block_reduce<1, true>(mx, R);
    const double ct = 1.0 / limit_scaling(fmax(sum[0] / double(n), limit_scaling(mx[0])));
    for (int k = tid; k < P.nnz_p; k += T) W.Pval[k] *= ct;
    for (int j = tid; j < n; j += T) W.q[j] *= ct;
    c *= ct;
    __syncthreads();
  }
  const double cinv = 1.0 / c;

  // ---- scaled bounds, constraint types, rho vector (set_rho_vec) ---------------------------
  double rho = fmin(fmax(S.rho, kRhoMin), kRhoMax);
  for (int i = tid; i < m; i += T) {
    const double lo = W.l[i] * W.E[i], hi = W.u[i] * W.E[i];
    W.l[i] = lo; W.u[i] = hi;
    const signed char ct = constraint_type(lo, hi);
    W.ctype[i] = ct;
    W.rho[i] = ct == -1 ? kRhoMin : (ct == 1 ? kRhoEqOverIneq * rho : rho);
  }
  __syncthreads();
  build_preconditioner(P, W, sigma, S.pcg_precond);

  const PatternOps I{P};
  const int interval = rho_interval(S);
  const double pcg_tol2 = S.pcg_tol * S.pcg_tol;
  int status = OCP_B200_QP_UNSOLVED, iter = 0, pcg_total = 0, rho_updates = 0, checks = 0, n_trace = 0;
  double prim_res = 0.0, dual_res = 0.0;
  bool done = false;

  for (iter = 1; iter <= S.admm_max_iter && !done; ++iter) {
    // ---- reduced KKT right-hand side and initial CG residual -------------------------------
    // b = sigma x - q + A'(rho z - y);  r = b - K xt, with zt = A xt kept up to date
    for (int i = tid; i < m; i += T) {
      const double rh = W.rho[i];
      W.w[i] = rh * W.z[i] - W.y[i];
      W.t[i] = rh * W.zt[i];
    }
    __syncthreads();
    double nb[2] = {0.0, 0.0};
    for (int j = tid; j < n; j += T) {
      const double b = sigma * W.x[j] - W.q[j] + col_dot_A(P, W.Aval, W.w, j);
      const double kx = sigma * W.xt[j] + col_dot_P(P, W.Pval, W.xt, j) + col_dot_A(P, W.Aval, W.t, j);
      const double r = b - kx;
      W.r[j] = r;
      nb[0] += b * b;
      nb[1] += r * r;
    }
    block_reduce<2, false>(nb, R);
    const double stop2 = pcg_tol2 * nb[0];
    double rr = nb[1];
    if (rr > stop2 && rr > 0.0) {
      double rz1[1] = {apply_preconditioner(P, W, S.pcg_precond)};
      for (int j = tid; j < n; j += T) W.d[j] = W.zc[j];
      block_reduce<1, false>(rz1, R);
      double rz = rz1[0];
      for (int k = 0; k < S.pcg_max_iter; ++k) {
        // t = A d, w = rho .* t
        for_rows_A(P, W.Aval, W.d, [&](int i, double s) { W.t[i] = s; W.w[i] = W.rho[i] * s; });
        __syncthreads();
        double dkd[1] = {0.0};
        for (int j = tid; j < n; j += T) {
          const double dj = W.d[j];
          const double kd = sigma * dj + col_dot_P(P, W.Pval, W.d, j) + col_dot_A(P, W.Aval, W.w, j);
          W.Kd[j] = kd;
          dkd[0] += dj * kd;
        }
        block_reduce<1, false>(dkd, R);
        const double alpha = rz / dkd[0];
        for (int j = tid; j < n; j += T) { W.xt[j] += alpha * W.d[j]; W.r[j] -= alpha * W.Kd[j]; }
        for (int i = tid; i < m; i += T) W.zt[i] += alpha * W.t[i];
        ++pcg_total;
        __syncthreads();
        double v2[2];
        v2[0] = apply_preconditioner(P, W, S.pcg_precond);
        v2[1] = 0.0;
        for (int j = tid; j < n; j += T) v2[1] += W.r[j] * W.r[j];
        block_reduce<2, false>(v2, R);
        rr = v2[1];
        if (!(rr > stop2)) break;
        const double beta = v2[0] / rz;
        rz = v2[0];
        for (int j = tid; j < n; j += T) W.d[j] = W.zc[j] + beta * W.d[j];
        __syncthreads();
      }
    }
    __syncthreads();

    // ---- x, z, y updates with relaxation and projection (update_x / update_z / update_y) ----
    for (int i = tid; i < m; i += T) {
      const double zr = relax * W.zt[i] + (1.0 - relax) * W.z[i];
      const double rinv = 1.0 / W.rho[i];
      const double zn = fmin(fmax(zr + rinv * W.y[i], W.l[i]), W.u[i]);
      const double dy = W.rho[i] * (zr - zn);
      W.y[i] += dy;
      W.z[i] = zn;
      W.dy[i] = dy;
    }
    for (int j = tid; j < n; j += T) {
      const double xn = relax * W.xt[j] + (1.0 - relax) * W.x[j];
      W.dx[j] = xn - W.x[j];
      W.x[j] = xn;
    }
    __syncthreads();

    const IterFlags F(S, interval, iter);
    if (!F.want_info()) continue;

    // ---- update_info, check_termination, adapt_rho (admm_common.cuh) -------------------------
    ++checks;
    const QpVec V = qp_vectors(W, n, m);
    double mx[kRedWidth];
    update_info(I, V, R, mx);
    prim_res = prim_residual(mx);
    dual_res = dual_residual(mx, cinv);
    if (F.can_check || F.last_iter) {
      const int st = check_termination(I, V, S, R, mx, c, cinv);
      if (F.can_check) record_trace(A, inst, n_trace, iter, prim_res, dual_res, rho, pcg_total, st);
      if (st >= 0) { status = st; done = true; continue; }
      if (F.last_iter) { status = approximate_status(S, mx, cinv); done = true; continue; }
    }
    if (F.rho_time && adapt_rho(S, mx, rho)) {
      ++rho_updates;
      for (int i = tid; i < m; i += T) {
        const signed char ct = W.ctype[i];
        W.rho[i] = ct == -1 ? kRhoMin : (ct == 1 ? kRhoEqOverIneq * rho : rho);
      }
      __syncthreads();
      build_preconditioner(P, W, sigma, S.pcg_precond);
    }
  }
  if (!done) status = OCP_B200_QP_MAX_ITER_REACHED;
  if (A.trace && inst == 0 && tid == 0 && A.n_trace) *A.n_trace = n_trace;
  out = QpResult{status, done ? iter - 1 : S.admm_max_iter, pcg_total, rho_updates, checks, prim_res, dual_res, rho};
  store_solution(qp_vectors(W, n, m), status, cinv);
}

// persistent kernel: CTAs pull instances from A.counter
template <bool kResident>
__global__ void __launch_bounds__(512, 1)
admm_solve_kernel(const PatternDev P, const ocp_b200_settings S, const SolveArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red_buf[2 * kMaxWarps * kRedWidth];
  __shared__ int s_inst;
  Work W;
  PatternDev PL = P;
  if (kResident) {
    double* base = reinterpret_cast<double*>(smem_raw);
    carve(W, base, P);
    // index structures move into shared memory once per CTA (staged_idx_entries sizes this list)
    idx_t* ip = reinterpret_cast<idx_t*>(base + work_doubles(P));
    auto stage = [&](const idx_t*& ptr, int count) {
      const idx_t* src = ptr;
      for (int k = threadIdx.x; k < count; k += blockDim.x) ip[k] = src[k];
      ptr = ip;
      ip += (count + 7) & ~7;
    };
    stage(PL.a_colptr, P.n + 1); stage(PL.a_rowidx, P.nnz_a); stage(PL.a_rowptr, P.m + 1);
    stage(PL.a_colidx, P.nnz_a); stage(PL.a_perm, P.nnz_a); stage(PL.p_colptr, P.n + 1);
    stage(PL.p_rowidx, P.nnz_p); stage(PL.blk_ptr, P.nblk + 1); stage(PL.blk_of_col, P.n);
    stage(PL.rows_long, P.n_long); stage(PL.rows_short, P.n_short);
    __syncthreads();
  } else {
    carve(W, A.slab + size_t(blockIdx.x) * A.slab_doubles, P);
  }
  Reducer R{red_buf, 0, kMaxWarps * kRedWidth};
  for (int inst; (inst = next_instance(A, s_inst)) < A.B;) {
    QpResult res;
    solve_instance(PL, S, A, W, R, inst, res);
    write_outputs(P, A, W.x, W.y, R, inst, res);
  }
}

}  // namespace pcg
}  // namespace ocpb200
