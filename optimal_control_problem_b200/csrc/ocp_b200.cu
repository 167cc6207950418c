// ocp_b200.cu -- implementation of the C ABI in include/ocp_b200.h.
//
// Host side of the B200 CUDA_SQP path: owns the device copies of the index structures,
// the per-batch QP buffers and the stage library, and drives the SQP loop
// (SQPOptimizationSolver.cpp:127-216 of the reference) as a fixed launch sequence
//   for step in 0..step_num-1:  assemble (stage library)  ->  admm_solve_kernel (+ x update)
//   objective (stage library) -> store_objective
// with no host round trip between the launches.  There is no CPU path in this file: without
// a CUDA device every entry point that computes returns OCP_B200_ERR_NO_DEVICE.
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "admm_pcg_kernel.cuh"
#include "compact_launch.h"
#include "direct_launch.h"
#include "direct_layout.cuh"
#include "ocp_b200_model.h"

namespace ocpb200 {
// f -> stats column, after the objective kernel of the stage library has run
// receding-horizon shift of the iterates: frame k <- frame k+1 (k < H-1), last frame repeated.
// One CTA per instance; the row is staged in shared memory so the shift is in place.
__global__ void shift_iterate_kernel(int nf, int N, double* __restrict__ x) {
  extern __shared__ double row[];
  double* xi = x + static_cast<size_t>(blockIdx.x) * N;
  for (int j = threadIdx.x; j < N; j += blockDim.x) row[j] = xi[j];
  __syncthreads();
  for (int j = threadIdx.x; j < N; j += blockDim.x) xi[j] = row[j + nf < N ? j + nf : j];
}

__global__ void store_objective_kernel(int B, const double* __restrict__ f, double* __restrict__ stats) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) stats[size_t(b) * OCP_B200_NSTATS + OCP_B200_STAT_OBJECTIVE] = f[b];
}

}  // namespace ocpb200

namespace {

thread_local std::string g_error;

int fail(int code, const std::string& msg) {
  g_error = msg;
  return code;
}

#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (expr);                                                                   \
    if (e_ != cudaSuccess)                                                                     \
      return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver ? OCP_B200_ERR_NO_DEVICE \
                                                                               : OCP_B200_ERR_CUDA, \
                  std::string(#expr) + ": " + cudaGetErrorString(e_));                         \
  } while (0)

#define RC_TRY(expr) do { int rc_ = (expr); if (rc_ != OCP_B200_OK) return rc_; } while (0)

// Every entry point works on the handle's device and puts the caller's current device back when it returns
// (the caller may be a torch process whose current device is another GPU).
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  cudaError_t enter(int dev) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev != dev) { e = cudaSetDevice(dev); changed = e == cudaSuccess; }
    return e;
  }
  ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};
#define ENTER_DEVICE(dev) DeviceGuard device_guard_; CUDA_TRY(device_guard_.enter(dev))

using ocpb200::idx_t;
using ocpb200::PatternDev;
using ocpb200::SolveArgs;

typedef const ocp_b200_model_info* (*model_info_fn)(void);
typedef int (*model_assemble_fn)(int, const double*, const double*, const double*, const double*, const double*,
                                 const double*, const double*, double*, int, double*, int, double*, int, double*,
                                 double*, int, void*);
typedef int (*model_objective_fn)(int, const double*, const double*, double*, void*);

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t count) {
    if (count <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&p), std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) cap = count;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// rows with at least kLongRow entries are handled by four lanes each in the row-wise products, the others by one
// thread.  Measured (quadrotor, rows of <= 17 entries): one thread per row beats four lanes per row by 7 %.
constexpr int kLongRow = 64;
// slots of the block staging ring: the one-CTA/SM slab plan (PLACE_BIG) takes kStageSlots when shared memory allows
constexpr int kStageSlots = 8, kStageSlotsMin = 4;

}  // namespace

// One launch configuration of the ADMM solve.  place: -1 the PCG kernel, 0-3 the direct kernel under that
// ocpb200::direct::Placement, 4 the compact kernel.
struct LaunchPlan {
  int place = -1, threads = 0, smem_bytes = 0, max_ctas = 1;
  uint32_t smem_mask = 0;    // direct kernel: which state arrays live in shared memory
  int compact_flags = 0;     // compact kernel: which streamed vectors moved into shared memory
  size_t slab_doubles = 0;   // per-CTA global slab
};

struct ocp_b200_solver {
  // problem
  int np = 0, nf = 0, horizon = 0, ng = 0, n = 0, m = 0, N = 0, nnz_h = 0, nnz_a = 0, nnz_p = 0;
  int device = 0;
  std::vector<int> h_colptr, h_rowidx, a_colptr, a_rowidx;
  ocp_b200_settings settings;
  // device index structures
  PatternDev pat{};
  DevBuf<idx_t> d_idx;
  DevBuf<int> d_int;
  DevBuf<ocpb200::KEntry> d_kent;
  DevBuf<ocpb200::KRun> d_krun;
  // stage-periodic templates of the index structures (compact throughput kernel); compact_ok: they exist
  DevBuf<uint32_t> d_arena;
  ocpb200::CompactIdx cidx{};
  int compact_ok = 0;
  // stage library
  void* lib = nullptr;
  model_assemble_fn assemble = nullptr;
  model_objective_fn objective = nullptr;
  // launch configuration
  int num_sms = 0;
  LaunchPlan deep, wide;       // latency plan (batches of at most one instance per SM) and throughput plan
  // workspaces (device)
  DevBuf<double> hv, q, av, l, u, solx, soly, info, slab, trace;
  DevBuf<double> x, p, frames, lbx, ubx, lbg, ubg, f, stats;
  DevBuf<int> counter;
  DevBuf<long long> phase;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  // optional per-kernel timing (ocp_b200_set_profiling): event pairs around every launch
  int profiling = 0;
  std::vector<cudaEvent_t> ev;      // pairs: start, stop
  std::vector<int> ev_kind;         // OCP_B200_PROF_* of each pair
  double prof_ms[OCP_B200_NPROF] = {0, 0, 0};
  long long prof_count[OCP_B200_NPROF] = {0, 0, 0};
};

namespace {

int upload_pattern(ocp_b200_solver* s, int num_blocks, const int* block_ptr) {
  const int n = s->n, m = s->m;
  const std::vector<int>&ac = s->a_colptr, &ar = s->a_rowidx, &hc = s->h_colptr, &hr = s->h_rowidx;
  // CSR view of A with the permutation back to CSC positions
  std::vector<int> rowptr(m + 1, 0), colidx(s->nnz_a), perm(s->nnz_a);
  for (int k = 0; k < s->nnz_a; ++k) rowptr[ar[k] + 1]++;
  for (int i = 0; i < m; ++i) rowptr[i + 1] += rowptr[i];
  {
    std::vector<int> next(rowptr.begin(), rowptr.end() - 1);
    for (int j = 0; j < n; ++j)
      for (int k = ac[j]; k < ac[j + 1]; ++k) { const int t = next[ar[k]]++; colidx[t] = j; perm[t] = k; }
  }
  // P: full symmetric pattern mirrored from the UPPER triangle of H (OsqpEigen hands OSQP the
  // upper triangle only); p_src = position of the upper-triangle twin in the caller's values
  std::vector<std::vector<std::pair<int, int>>> cols(n);
  for (int j = 0; j < n; ++j)
    for (int k = hc[j]; k < hc[j + 1]; ++k) {
      const int i = hr[k];
      if (i > j) continue;
      cols[j].push_back({i, k});
      if (i != j) cols[i].push_back({j, k});
    }
  std::vector<int> pc(n + 1, 0), pr, psrc;
  for (int j = 0; j < n; ++j) {
    std::sort(cols[j].begin(), cols[j].end());
    for (auto& e : cols[j]) { pr.push_back(e.first); psrc.push_back(e.second); }
    pc[j + 1] = static_cast<int>(pr.size());
  }
  s->nnz_p = static_cast<int>(pr.size());
  // preconditioner blocks
  std::vector<int> blk;
  if (num_blocks > 0 && block_ptr) {
    blk.assign(block_ptr, block_ptr + num_blocks + 1);
    if (blk.front() != 0 || blk.back() != n) return fail(OCP_B200_ERR_INVALID, "block_ptr must run from 0 to n");
    for (int b = 0; b < num_blocks; ++b)
      if (blk[b + 1] <= blk[b]) return fail(OCP_B200_ERR_INVALID, "block_ptr must be strictly ascending");
  } else {
    // default: [p | frame 0 | ... | frame H-1]; blocks wider than 64 columns (a QP-only handle
    // is one "frame") are cut into 32-column pieces
    std::vector<int> cuts{0};
    if (s->np > 0) cuts.push_back(s->np);
    for (int k = 0; k < s->horizon; ++k) cuts.push_back(s->np + (k + 1) * s->nf);
    blk.push_back(0);
    for (size_t b = 0; b + 1 < cuts.size(); ++b) {
      if (cuts[b + 1] - cuts[b] > 64)
        for (int j = cuts[b] + 32; j < cuts[b + 1]; j += 32) blk.push_back(j);
      blk.push_back(cuts[b + 1]);
    }
  }
  const int nblk = static_cast<int>(blk.size()) - 1;
  std::vector<int> blk_of(n), minv_off(nblk);
  int minv = 0, max_bs = 0;
  for (int b = 0; b < nblk; ++b) {
    const int bs = blk[b + 1] - blk[b];
    minv_off[b] = minv;
    minv += bs * bs;
    max_bs = std::max(max_bs, bs);
    for (int j = blk[b]; j < blk[b + 1]; ++j) blk_of[j] = b;
  }
  // Gauss-Jordan on large dense blocks is pointless (and the block store would not fit):
  // fall back to Jacobi for such partitions
  if (max_bs > 64) return fail(OCP_B200_ERR_UNSUPPORTED, "preconditioner blocks larger than 64 columns are not supported");
  std::vector<int> rows_long, rows_short;
  for (int i = 0; i < m; ++i) (rowptr[i + 1] - rowptr[i] >= kLongRow ? rows_long : rows_short).push_back(i);

  if (n + 1 > 65535 || m + 1 > 65535 || s->nnz_a > 65535 || s->nnz_p > 65535)
    return fail(OCP_B200_ERR_UNSUPPORTED, "problem too large for 16-bit index structures (n, m, nnz < 65536)");

  // one idx_t arena, every array padded to 8 entries so that the shared-memory copy keeps alignment
  std::vector<idx_t> arena;
  auto push = [&](const std::vector<int>& v) {
    const size_t off = arena.size();
    for (int x : v) arena.push_back(static_cast<idx_t>(x));
    while (arena.size() % 8) arena.push_back(0);
    return off;
  };
  const size_t o_acp = push(ac), o_ari = push(ar), o_arp = push(rowptr), o_aci = push(colidx), o_perm = push(perm),
               o_pcp = push(pc), o_pri = push(pr), o_rl = push(rows_long), o_rs = push(rows_short);
  const size_t direct_entries = arena.size();   // what the direct kernel stages in shared memory
  const size_t o_blk = push(blk), o_bof = push(blk_of);   // PCG kernel only
  CUDA_TRY(s->d_idx.reserve(arena.size()));
  CUDA_TRY(cudaMemcpy(s->d_idx.p, arena.data(), arena.size() * sizeof(idx_t), cudaMemcpyHostToDevice));
  std::vector<int> iarena(psrc);
  const size_t o_minv = iarena.size();
  iarena.insert(iarena.end(), minv_off.begin(), minv_off.end());
  CUDA_TRY(s->d_int.reserve(iarena.size()));
  CUDA_TRY(cudaMemcpy(s->d_int.p, iarena.data(), iarena.size() * sizeof(int), cudaMemcpyHostToDevice));

  PatternDev& P = s->pat;
  P.n = n; P.m = m; P.nnz_a = s->nnz_a; P.nnz_p = s->nnz_p; P.nnz_h = s->nnz_h;
  P.nblk = nblk; P.minv_doubles = std::max(minv, n); P.max_bs = max_bs;
  P.n_long = static_cast<int>(rows_long.size()); P.n_short = static_cast<int>(rows_short.size());
  const idx_t* base = s->d_idx.p;
  P.a_colptr = base + o_acp; P.a_rowidx = base + o_ari; P.a_rowptr = base + o_arp; P.a_colidx = base + o_aci;
  P.a_perm = base + o_perm; P.p_colptr = base + o_pcp; P.p_rowidx = base + o_pri; P.blk_ptr = base + o_blk;
  P.blk_of_col = base + o_bof; P.rows_long = base + o_rl; P.rows_short = base + o_rs;
  P.p_src = s->d_int.p; P.minv_off = s->d_int.p + o_minv;

  P.idx_entries = static_cast<int>(direct_entries);
  P.idx_base = base;

  // bordered block-tridiagonal structure of K for the direct kernel: border = the np parameter
  // columns, blocks = groups of G consecutive stages (G the largest divisor of the horizon that
  // keeps a block at <= 20 columns, so that long horizons of small stages take fewer
  // sequential block steps)
  {
    int G = 1;
    for (int g = 1; g <= s->horizon; ++g)
      if (s->horizon % g == 0 && g * s->nf <= 20) G = g;
    const int bs = G * s->nf, nb = s->horizon / G;
    P.tri_np = s->np; P.tri_bs = bs; P.tri_nb = nb; P.tri_ld = (bs + 2) & ~1;   // even pitch: 16-byte aligned block rows
    bool ok = bs <= 64 && s->np <= 64;
    auto blk_of_col = [&](int j) { return j < s->np ? -1 : (j - s->np) / bs; };
    for (int j = 0; j < n && ok; ++j)
      for (int k = pc[j]; k < pc[j + 1]; ++k) {
        const int bi = blk_of_col(pr[k]), bj = blk_of_col(j);
        if (bi >= 0 && bj >= 0 && std::abs(bi - bj) > 1) { ok = false; break; }
      }
    for (int i = 0; i < m && ok; ++i) {
      int lo = 1 << 30, hi = -1;
      for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
        const int bj = blk_of_col(colidx[k]);
        if (bj >= 0) { lo = std::min(lo, bj); hi = std::max(hi, bj); }
      }
      if (hi >= 0 && hi - lo > 1) ok = false;
    }
    P.tri_ok = ok ? 1 : 0;
    P.kprog_entries = 0; P.kprog = nullptr; P.kruns = nullptr;
    if (ok) {
      // K-assembly program: every element of the factor storage that can be non-zero
      const int ld = P.tri_ld, N = nb * bs, np = s->np;
      std::vector<ocpb200::KEntry> ents;
      std::vector<ocpb200::KRun> runs;
      auto add = [&](int i, int j, uint32_t d0, uint32_t d1) {
        ocpb200::KEntry e{};
        e.dest0 = d0; e.dest1 = d1; e.ppos = -1; e.run_begin = static_cast<uint32_t>(runs.size()); e.nruns = 0;
        e.diag = i == j ? 1 : 0; e.pad = 0;
        for (int k = pc[j]; k < pc[j + 1]; ++k)
          if (pr[k] == i) { e.ppos = k; break; }
        int ka = ac[i], kc = ac[j];
        const int ea = ac[i + 1], ec = ac[j + 1];
        while (ka < ea && kc < ec) {
          if (ar[ka] == ar[kc]) {
            if (e.nruns > 0 && runs.back().ka + runs.back().len == ka && runs.back().kc + runs.back().len == kc &&
                runs.back().row0 + runs.back().len == ar[ka]) {
              runs.back().len++;
            } else {
              runs.push_back({static_cast<uint16_t>(ka), static_cast<uint16_t>(kc), 1, static_cast<uint16_t>(ar[ka])});
              e.nruns++;
            }
            ++ka; ++kc;
          } else if (ar[ka] < ar[kc]) ++ka;
          else ++kc;
        }
        if (e.nruns > 0 || e.ppos >= 0 || e.diag) ents.push_back(e);
      };
      const uint32_t none = 0xffffffffu;
      auto dst = [](uint32_t arr, size_t off) { return (arr << 30) | static_cast<uint32_t>(off); };
      bool fits = size_t(nb) * bs * ld < (1u << 30) && size_t(np) * N < (1u << 30);
      if (fits) {
        for (int k = 0; k < nb; ++k)
          for (int r = 0; r < bs; ++r)
            for (int c = r; c < bs; ++c)
              add(np + k * bs + r, np + k * bs + c, dst(0, size_t(k) * bs * ld + r * ld + c),
                  r == c ? none : dst(0, size_t(k) * bs * ld + c * ld + r));
        for (int k = 1; k < nb; ++k)
          for (int r = 0; r < bs; ++r)
            for (int c = 0; c < bs; ++c)
              add(np + k * bs + r, np + (k - 1) * bs + c, dst(1, size_t(k) * bs * ld + r * ld + c), none);
        for (int r = 0; r < np; ++r)
          for (int j = 0; j < N; ++j) add(r, np + j, dst(2, size_t(r) * N + j), none);
        for (int r = 0; r < np; ++r)
          for (int c = r; c < np; ++c)
            add(r, c, dst(3, size_t(r) * (np + 1) + c), r == c ? none : dst(3, size_t(c) * (np + 1) + r));
        // longest entries first: threads take entries round-robin, so the tail stays short
        std::stable_sort(ents.begin(), ents.end(), [&](const ocpb200::KEntry& a, const ocpb200::KEntry& b) {
          auto len = [&](const ocpb200::KEntry& e) { int t = 0; for (int q = 0; q < e.nruns; ++q) t += runs[e.run_begin + q].len; return t; };
          return len(a) > len(b);
        });
        CUDA_TRY(s->d_kent.reserve(ents.size()));
        CUDA_TRY(s->d_krun.reserve(runs.size()));
        CUDA_TRY(cudaMemcpy(s->d_kent.p, ents.data(), ents.size() * sizeof(ocpb200::KEntry), cudaMemcpyHostToDevice));
        if (!runs.empty())
          CUDA_TRY(cudaMemcpy(s->d_krun.p, runs.data(), runs.size() * sizeof(ocpb200::KRun), cudaMemcpyHostToDevice));
        P.kprog_entries = static_cast<int>(ents.size());
        P.kprog = s->d_kent.p; P.kruns = s->d_krun.p;
      }
    }
  }
  // stage-periodic templates of the CSC / CSR structures of A and of the symmetrised P (periodic_index.h)
  s->compact_ok = 0;
  if (P.tri_ok && P.kprog_entries > 0 && rows_long.empty()) {
    std::vector<int> periods;
    for (int p = 1; p <= 96; ++p) periods.push_back(p);
    ocpb200::PIndexHost hc, hr, hp;
    const bool built = ocpb200::build_periodic_index(ac, ar, {}, periods, hc) &&
                       ocpb200::build_periodic_index(rowptr, colidx, perm, periods, hr) &&
                       ocpb200::build_periodic_index(pc, pr, {}, periods, hp);
    const size_t maxreg = std::max({hc.reg.size(), hr.reg.size(), hp.reg.size()});
    if (built && maxreg <= size_t(ocpb200::kMaxDevRegions)) {
      std::vector<uint32_t> arena32;
      auto place = [&](const ocpb200::PIndexHost& h, ocpb200::PIndexDev& d) {
        d.nreg = static_cast<int>(h.reg.size());
        for (int r = 0; r < ocpb200::kMaxDevRegions; ++r) {
          d.ibound[r] = r < d.nreg ? h.reg[r].i1 : 0x7fffffff;
          d.kbound[r] = r < d.nreg ? h.reg[r].k1 : 0x7fffffff;
        }
        d.reg_off = static_cast<int>(arena32.size());
        const uint32_t* rw = reinterpret_cast<const uint32_t*>(h.reg.data());
        arena32.insert(arena32.end(), rw, rw + h.reg.size() * (sizeof(ocpb200::PRegion) / 4));
        d.tptr_off = static_cast<int>(arena32.size());
        arena32.insert(arena32.end(), h.tptr.begin(), h.tptr.end());
        d.tent_off = static_cast<int>(arena32.size());
        arena32.insert(arena32.end(), h.tent.begin(), h.tent.end());
        d.tent2_off = h.tent2.empty() ? -1 : static_cast<int>(arena32.size());
        arena32.insert(arena32.end(), h.tent2.begin(), h.tent2.end());
      };
      place(hc, s->cidx.acol); place(hr, s->cidx.arow); place(hp, s->cidx.pcol);
      CUDA_TRY(s->d_arena.reserve(arena32.size()));
      CUDA_TRY(cudaMemcpy(s->d_arena.p, arena32.data(), arena32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
      s->cidx.arena = s->d_arena.p;
      s->cidx.arena_words = static_cast<int>(arena32.size());
      s->compact_ok = 1;
    }
  }
  return OCP_B200_OK;
}

// Chooses the kernel for the current settings and lays out its per-instance state: shared
// memory first, the rest in a per-CTA global slab.
int plan_launch(ocp_b200_solver* s) {
  const PatternDev& P = s->pat;
  int max_optin = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, s->device));
  if (s->settings.pcg_precond != OCP_B200_PRECOND_BLOCK_TRIDIAG || !P.tri_ok) {
    // PCG kernel, one plan for every batch size: its state in shared memory when it fits ("resident"), else in the slab
    LaunchPlan L;
    L.threads = 512;
    const size_t want = ocpb200::pcg::work_doubles(P) * sizeof(double) + ocpb200::pcg::staged_idx_entries(P) * sizeof(idx_t);
    cudaFuncAttributes fa{};
    CUDA_TRY(cudaFuncGetAttributes(&fa, ocpb200::pcg::admm_solve_kernel<true>));
    int per_sm = 1;
    if (want <= size_t(max_optin) - fa.sharedSizeBytes) {
      L.smem_bytes = static_cast<int>(want);
      CUDA_TRY(cudaFuncSetAttribute(ocpb200::pcg::admm_solve_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    max_optin - static_cast<int>(fa.sharedSizeBytes)));
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ocpb200::pcg::admm_solve_kernel<true>, L.threads,
                                                             L.smem_bytes));
    } else {
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ocpb200::pcg::admm_solve_kernel<false>, L.threads, 0));
    }
    // reported for the resident kernel as well, although it launches without a slab
    L.slab_doubles = (ocpb200::pcg::work_doubles(P) + 15) & ~size_t(15);
    L.max_ctas = std::max(1, per_sm) * s->num_sms;
    s->deep = s->wide = L;
    return OCP_B200_OK;
  }
  namespace D = ocpb200::direct;
  // Two plans are kept.  `wide`: 2 CTAs per SM (vectors, A values, index arrays and scratch in
  // shared memory, factor blocks in an L2-resident slab) -- the throughput plan, used when the
  // batch has more instances than SMs.  `deep`: 1 CTA per SM with as much state as fits in shared
  // memory (everything, for the H=20 quadrotor) -- the latency plan, used for small batches.
  // OCP_B200_PLAN = smem | multi | mixed forces one of them (diagnostics).
  const char* env = std::getenv("OCP_B200_PLAN");
  const bool force_stream = std::getenv("OCP_B200_FORCE_STREAM") != nullptr;
  auto smem_bytes = [&](int place) { return D::plan_state(P, place, 0, false).smem_doubles * sizeof(double); };
  s->pat.stage_slots = kStageSlotsMin;
  auto make_plan = [&](int place, LaunchPlan& L) -> int {
    D::KernelInfo kx{};
    const D::EntryPoints& ep = D::entry_points(place);
    CUDA_TRY(ep.kernel_info(&kx));
    CUDA_TRY(ep.set_max_dynamic_smem(max_optin - kx.static_smem));
    const D::StateLayout st = D::plan_state(P, place, (size_t(max_optin) - kx.static_smem) / sizeof(double), force_stream);
    const int bytes = static_cast<int>(st.smem_doubles * sizeof(double));
    int occ = 1;
    CUDA_TRY(ep.occupancy(bytes, &occ));
    L = LaunchPlan{place, kx.threads, bytes, std::max(1, occ) * s->num_sms, st.mask, 0, st.slab_doubles};
    return OCP_B200_OK;
  };
  D::KernelInfo ki{}, km{}, kb{};
  CUDA_TRY(D::kSmem.kernel_info(&ki));
  CUDA_TRY(D::kMulti.kernel_info(&km));
  CUDA_TRY(D::kBig.kernel_info(&kb));
  const bool fits_all = smem_bytes(D::PLACE_SMEM) + ki.static_smem <= size_t(max_optin);
  const bool fits_multi = (smem_bytes(D::PLACE_MULTI) + km.static_smem + 1024) * 2 <= size_t(228) * 1024;
  const bool fits_big = smem_bytes(D::PLACE_BIG) + kb.static_smem <= size_t(max_optin);
  const bool forced_big = env && !std::strcmp(env, "big");
  if (fits_big && ((!fits_all && !fits_multi) || forced_big)) {
    // the 1-CTA/SM slab plan is the only one: widen the staging area to a ring of 4 blocks per
    // sweep chain (asynchronous bulk copies, tri_twisted.cuh) when shared memory allows
    s->pat.stage_slots = kStageSlots;
    if (smem_bytes(D::PLACE_BIG) + kb.static_smem > size_t(max_optin)) s->pat.stage_slots = kStageSlotsMin;
  }
  int deep = fits_all ? 1 : (fits_big ? 3 : 0), wide = fits_multi ? 2 : deep;
  if (env && !std::strcmp(env, "multi") && fits_multi) deep = wide = 2;
  else if (env && !std::strcmp(env, "mixed")) deep = wide = 0;
  else if (env && !std::strcmp(env, "smem") && fits_all) deep = wide = 1;
  else if (env && !std::strcmp(env, "big") && fits_big) deep = wide = 3;
  RC_TRY(make_plan(deep, s->deep));
  RC_TRY(make_plan(wide, s->wide));
  // compact throughput plan (admm_compact_kernel.cuh): index templates, streamed slab vectors, four CTAs per SM --
  // taken when it keeps more threads resident than the plan above (OCP_B200_PLAN=compact forces it, any other value
  // of OCP_B200_PLAN keeps it out).  q, then l and u, move from the slab into shared memory while the residency
  // target still holds.
  if (s->compact_ok && (P.tri_bs == 16 || P.tri_bs == 20) && P.tri_ld == P.tri_bs + 2 && (!env || !std::strcmp(env, "compact"))) {
    namespace K = ocpb200::compact;
    D::KernelInfo kc{};
    CUDA_TRY(K::kernel_info(P.tri_bs, &kc));
    CUDA_TRY(K::set_max_dynamic_smem(P.tri_bs, max_optin - kc.static_smem));
    int best_flags = -1, best_occ = 0;
    size_t best_sm = 0, best_sl = 0;
    for (int flags : {3, 1, 0}) {   // most shared memory first
      size_t sm_d = 0, sl_d = 0;
      bool lay_ok = false;
      K::plan_sizes(P, s->cidx.arena_words, flags, &sm_d, &sl_d, &lay_ok);
      if (!lay_ok || sm_d * sizeof(double) + kc.static_smem > size_t(max_optin)) continue;
      // residency by hand: the occupancy calculator answers 1 for a kernel that allocates Tensor Memory (it cannot know
      // how many of the 512 columns a CTA will ask for); the compact kernel takes 128 of them when BS == 16
      int occ = 0;
      {
        int smem_sm = 0, regs_sm = 0;
        CUDA_TRY(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, s->device));
        CUDA_TRY(cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, s->device));
        const int regs_cta = ((kc.regs + 7) / 8 * 8) * kc.threads;
        const size_t smem_cta = sm_d * sizeof(double) + kc.static_smem + 1024;   // 1 KB reserved per CTA
        occ = std::min({regs_sm / std::max(1, regs_cta), static_cast<int>(size_t(smem_sm) / smem_cta), 2048 / kc.threads,
                        P.tri_bs == 16 ? 512 / 128 : 32});
      }
      if (occ > best_occ && best_occ < K::kCtasPerSm) { best_occ = occ; best_flags = flags; best_sm = sm_d; best_sl = sl_d; }
    }
    if (best_flags >= 0) {
      const int occ = std::min(best_occ, K::kCtasPerSm);
      if (occ * kc.threads > (s->wide.max_ctas / s->num_sms) * s->wide.threads || env) {
        s->wide = LaunchPlan{4, kc.threads, static_cast<int>(best_sm * sizeof(double)), occ * s->num_sms, 0, best_flags, best_sl};
        if (env) s->deep = s->wide;
      }
    }
  }
  return OCP_B200_OK;
}

int load_model(ocp_b200_solver* s, const char* path) {
  s->lib = dlopen(path, RTLD_NOW | RTLD_LOCAL);
  if (!s->lib) return fail(OCP_B200_ERR_MODEL, std::string("cannot load stage library: ") + dlerror());
  model_info_fn info_fn = reinterpret_cast<model_info_fn>(dlsym(s->lib, "ocp_b200_model_get_info"));
  s->assemble = reinterpret_cast<model_assemble_fn>(dlsym(s->lib, "ocp_b200_model_assemble"));
  s->objective = reinterpret_cast<model_objective_fn>(dlsym(s->lib, "ocp_b200_model_objective"));
  if (!info_fn || !s->assemble || !s->objective)
    return fail(OCP_B200_ERR_MODEL, "stage library does not export the ocp_b200_model.h symbols");
  const ocp_b200_model_info* mi = info_fn();
  if (!mi || mi->abi_version != OCP_B200_MODEL_ABI_VERSION)
    return fail(OCP_B200_ERR_MODEL, "stage library ABI version mismatch");
  if (mi->np != s->np || mi->nf != s->nf || mi->horizon != s->horizon || mi->ng != s->ng || mi->nnz_h != s->nnz_h ||
      mi->nnz_a != s->nnz_a)
    return fail(OCP_B200_ERR_MODEL, "stage library was generated for a different problem shape");
  if (std::memcmp(mi->h_colptr, s->h_colptr.data(), sizeof(int) * (s->n + 1)) ||
      std::memcmp(mi->h_rowidx, s->h_rowidx.data(), sizeof(int) * s->nnz_h) ||
      std::memcmp(mi->a_colptr, s->a_colptr.data(), sizeof(int) * (s->n + 1)) ||
      std::memcmp(mi->a_rowidx, s->a_rowidx.data(), sizeof(int) * s->nnz_a))
    return fail(OCP_B200_ERR_MODEL, "stage library sparsity pattern differs from the problem description");
  return OCP_B200_OK;
}

int check_settings(const ocp_b200_settings* t) {
  if (!t) return fail(OCP_B200_ERR_INVALID, "settings is NULL");
  if (t->sqp_step_num < 0 || t->admm_max_iter < 1 || t->check_termination < 0 || t->scaling_iters < 0 ||
      t->pcg_max_iter < 1 || !(t->rho > 0) || !(t->sigma > 0) || !(t->relax > 0 && t->relax < 2) ||
      !(t->eps_abs >= 0) || !(t->eps_rel >= 0) || !(t->pcg_tol > 0) || t->pcg_precond < 0 ||
      t->pcg_precond > OCP_B200_PRECOND_BLOCK_TRIDIAG)
    return fail(OCP_B200_ERR_INVALID, "settings out of range");
  return OCP_B200_OK;
}

// event pair around one launch when profiling is on
struct ProfScope {
  ocp_b200_solver* s; cudaStream_t st; cudaEvent_t stop = nullptr;
  ProfScope(ocp_b200_solver* s_, int kind, cudaStream_t st_) : s(s_), st(st_) {
    if (!s->profiling) return;
    // bounded: pairs that have completed are folded into the totals; with kMaxPending still in flight this
    // launch simply goes untimed (nothing blocks here)
    constexpr size_t kMaxPending = 4096;
    if (s->ev_kind.size() >= kMaxPending) {
      size_t keep = 0;
      for (size_t k = 0; k < s->ev_kind.size(); ++k) {
        cudaEvent_t ea = s->ev[2 * k], eb = s->ev[2 * k + 1];
        float t = 0.f;
        if (cudaEventQuery(eb) == cudaSuccess && cudaEventElapsedTime(&t, ea, eb) == cudaSuccess) {
          s->prof_ms[s->ev_kind[k]] += t; s->prof_count[s->ev_kind[k]]++;
          cudaEventDestroy(ea); cudaEventDestroy(eb);
        } else {
          s->ev[2 * keep] = ea; s->ev[2 * keep + 1] = eb; s->ev_kind[keep] = s->ev_kind[k]; ++keep;
        }
      }
      cudaGetLastError();
      s->ev.resize(2 * keep); s->ev_kind.resize(keep);
      if (keep >= kMaxPending) return;
    }
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
    s->ev.push_back(a); s->ev.push_back(b); s->ev_kind.push_back(kind);
    cudaEventRecord(a, st);
    stop = b;
  }
  ~ProfScope() { if (stop) cudaEventRecord(stop, st); }
};

// one ADMM launch over B instances
int launch_admm(ocp_b200_solver* s, SolveArgs& A, cudaStream_t st) {
  CUDA_TRY(s->counter.reserve(1));
  CUDA_TRY(cudaMemsetAsync(s->counter.p, 0, sizeof(int), st));
  A.counter = s->counter.p;
  A.phase = s->profiling >= 2 ? s->phase.p : nullptr;
  // small batches (at most one instance per SM): the latency plan; otherwise the throughput plan
  const LaunchPlan& L = A.B <= s->num_sms ? s->deep : s->wide;
  const int grid = std::min(A.B, L.max_ctas);
  ProfScope prof(s, OCP_B200_PROF_ADMM, st);
  // the resident PCG kernel (state in shared memory) takes no slab
  const bool slab = L.slab_doubles > 0 && (L.place >= 0 || L.smem_bytes == 0);
  A.slab = nullptr; A.slab_doubles = slab ? L.slab_doubles : 0;
  if (slab) {
    CUDA_TRY(s->slab.reserve(size_t(grid) * L.slab_doubles));
    A.slab = s->slab.p;
  }
  if (L.place < 0) {
    ocp_b200_settings t = s->settings;
    if (t.pcg_precond == OCP_B200_PRECOND_BLOCK_TRIDIAG) t.pcg_precond = OCP_B200_PRECOND_BLOCK_JACOBI;
    if (L.smem_bytes > 0) ocpb200::pcg::admm_solve_kernel<true><<<grid, L.threads, L.smem_bytes, st>>>(s->pat, t, A);
    else ocpb200::pcg::admm_solve_kernel<false><<<grid, L.threads, 0, st>>>(s->pat, t, A);
  } else if (L.place == 4) {
    CUDA_TRY(ocpb200::compact::launch(s->pat.tri_bs, grid, L.smem_bytes, st, s->pat, s->cidx, s->settings, A, L.compact_flags));
  } else {
    CUDA_TRY(ocpb200::direct::entry_points(L.place).launch(grid, L.smem_bytes, st, s->pat, s->settings, A, L.smem_mask));
  }
  CUDA_TRY(cudaGetLastError());
  s->launches++;
  return OCP_B200_OK;
}

int reserve_qp(ocp_b200_solver* s, int B) {
  CUDA_TRY(s->hv.reserve(size_t(B) * s->nnz_h));
  CUDA_TRY(s->q.reserve(size_t(B) * s->n));
  CUDA_TRY(s->av.reserve(size_t(B) * s->nnz_a));
  CUDA_TRY(s->l.reserve(size_t(B) * s->m));
  CUDA_TRY(s->u.reserve(size_t(B) * s->m));
  return OCP_B200_OK;
}

int assemble_on(ocp_b200_solver* s, int B, const double* x, const double* p, const double* frames,
                const double* lbx, const double* ubx, const double* lbg, const double* ubg, cudaStream_t st) {
  if (!s->assemble) return fail(OCP_B200_ERR_MODEL, "this handle has no stage library (QP-only handle)");
  ProfScope prof(s, OCP_B200_PROF_ASSEMBLE, st);
  const int rc = s->assemble(B, x, p, frames, lbx, ubx, lbg, ubg, s->hv.p, s->nnz_h, s->q.p, s->n, s->av.p,
                             s->nnz_a, s->l.p, s->u.p, s->m, st);
  if (rc != 0) return fail(OCP_B200_ERR_CUDA, std::string("stage assembly launch: ") +
                                                  cudaGetErrorString(static_cast<cudaError_t>(rc)));
  s->launches++;
  return OCP_B200_OK;
}

int h2d(double* dst, const double* src, size_t count, cudaStream_t st) {
  if (count == 0) return OCP_B200_OK;
  CUDA_TRY(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyHostToDevice, st));
  return OCP_B200_OK;
}
int d2h(double* dst, const double* src, size_t count, cudaStream_t st) {
  if (count == 0) return OCP_B200_OK;
  CUDA_TRY(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyDeviceToHost, st));
  return OCP_B200_OK;
}


int upload_problem_inputs(ocp_b200_solver* s, int B, const double* frames, const double* p, const double* lbx,
                          const double* ubx, const double* lbg, const double* ubg, cudaStream_t st) {
  CUDA_TRY(s->p.reserve(size_t(B) * s->np));
  CUDA_TRY(s->frames.reserve(size_t(B) * s->nf));
  CUDA_TRY(s->lbx.reserve(s->N)); CUDA_TRY(s->ubx.reserve(s->N));
  CUDA_TRY(s->lbg.reserve(s->ng)); CUDA_TRY(s->ubg.reserve(s->ng));
  RC_TRY(h2d(s->p.p, p, size_t(B) * s->np, st));
  if (frames) RC_TRY(h2d(s->frames.p, frames, size_t(B) * s->nf, st));
  RC_TRY(h2d(s->lbx.p, lbx, s->N, st)); RC_TRY(h2d(s->ubx.p, ubx, s->N, st));
  RC_TRY(h2d(s->lbg.p, lbg, s->ng, st)); RC_TRY(h2d(s->ubg.p, ubg, s->ng, st));
  return OCP_B200_OK;
}

}  // namespace

extern "C" {

void ocp_b200_default_settings(ocp_b200_settings* s) {
  if (!s) return;
  s->sqp_alpha = 0.1; s->sqp_step_num = 10;          // OptimalControlProblem.h:24-27
  s->eps_abs = 1e-3; s->eps_rel = 1e-3;              // SQPOptimizationSolver.cpp:83-84
  s->eps_prim_inf = 1e-4; s->eps_dual_inf = 1e-4;
  s->admm_max_iter = 10000;                          // SQPOptimizationSolver.cpp:85
  s->rho = 0.1; s->sigma = 1e-6; s->relax = 1.6;
  s->scaling_iters = 10; s->check_termination = 25;
  s->adaptive_rho = 1; s->adaptive_rho_interval = 0; s->adaptive_rho_tolerance = 5.0;
  s->pcg_max_iter = 500; s->pcg_tol = 1e-10; s->pcg_precond = OCP_B200_PRECOND_BLOCK_TRIDIAG;
}

int ocp_b200_abi_version(void) { return OCP_B200_ABI_VERSION; }
const char* ocp_b200_last_error(void) { return g_error.c_str(); }

int ocp_b200_create(const ocp_b200_problem_desc* d, const ocp_b200_settings* settings, ocp_b200_solver** out) {
  if (!d || !out) return fail(OCP_B200_ERR_INVALID, "desc/out is NULL");
  *out = nullptr;
  ocp_b200_settings dflt;
  if (!settings) { ocp_b200_default_settings(&dflt); settings = &dflt; }
  RC_TRY(check_settings(settings));
  // a QP-only handle (no stage library; CuCaQP) may have FEWER constraint rows than variables: ng = m - n < 0.
  // The OCP entry points need the identity rows of c = [p; x; g], i.e. ng >= 0.
  const bool qp_only = !(d->model_library && d->model_library[0]);
  if (d->np < 0 || d->nf <= 0 || d->horizon <= 0 || (d->ng < 0 && !qp_only) || !d->h_colptr || !d->a_colptr ||
      (d->nnz_h > 0 && !d->h_rowidx) || (d->nnz_a > 0 && !d->a_rowidx))
    return fail(OCP_B200_ERR_INVALID, "bad problem description");
  const long long n = (long long)d->np + (long long)d->nf * d->horizon, m = n + d->ng;
  if (m < 1) return fail(OCP_B200_ERR_INVALID, "a QP needs at least one constraint row (the reference's OSQP set-up rejects m = 0 as well)");
  if (n <= 0 || m > 65534) return fail(OCP_B200_ERR_UNSUPPORTED, "problem too large for 16-bit index structures");
  if (d->h_colptr[0] != 0 || d->h_colptr[n] != d->nnz_h || d->a_colptr[0] != 0 || d->a_colptr[n] != d->nnz_a)
    return fail(OCP_B200_ERR_INVALID, "column pointers do not match nnz");
  for (int j = 0; j < n; ++j) {
    if (d->h_colptr[j + 1] < d->h_colptr[j] || d->a_colptr[j + 1] < d->a_colptr[j])
      return fail(OCP_B200_ERR_INVALID, "column pointers must be non-decreasing");
    for (int k = d->h_colptr[j]; k < d->h_colptr[j + 1]; ++k)
      if (d->h_rowidx[k] < 0 || d->h_rowidx[k] >= n || (k > d->h_colptr[j] && d->h_rowidx[k] <= d->h_rowidx[k - 1]))
        return fail(OCP_B200_ERR_INVALID, "Hessian row indices must be strictly increasing within a column");
    for (int k = d->a_colptr[j]; k < d->a_colptr[j + 1]; ++k)
      if (d->a_rowidx[k] < 0 || d->a_rowidx[k] >= m || (k > d->a_colptr[j] && d->a_rowidx[k] <= d->a_rowidx[k - 1]))
        return fail(OCP_B200_ERR_INVALID, "Jacobian row indices must be strictly increasing within a column");
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(OCP_B200_ERR_NO_DEVICE, std::string("no CUDA device (there is no CPU fallback): ") +
                                            (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
  if (d->device < 0 || d->device >= ndev) return fail(OCP_B200_ERR_INVALID, "device ordinal out of range");
  ENTER_DEVICE(d->device);

  ocp_b200_solver* s = new (std::nothrow) ocp_b200_solver();
  if (!s) return fail(OCP_B200_ERR_INVALID, "out of host memory");
  s->np = d->np; s->nf = d->nf; s->horizon = d->horizon; s->ng = d->ng;
  s->n = static_cast<int>(n); s->m = static_cast<int>(m); s->N = d->nf * d->horizon;
  s->nnz_h = d->nnz_h; s->nnz_a = d->nnz_a; s->device = d->device;
  s->h_colptr.assign(d->h_colptr, d->h_colptr + n + 1); s->h_rowidx.assign(d->h_rowidx, d->h_rowidx + d->nnz_h);
  s->a_colptr.assign(d->a_colptr, d->a_colptr + n + 1); s->a_rowidx.assign(d->a_rowidx, d->a_rowidx + d->nnz_a);
  s->settings = *settings;
  auto bail = [&](int rc) { std::string keep = g_error; ocp_b200_destroy(s); g_error = keep; return rc; };
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, d->device) != cudaSuccess) return bail(fail(OCP_B200_ERR_CUDA, "cudaGetDeviceProperties failed"));
  if (prop.major < 10)
    return bail(fail(OCP_B200_ERR_UNSUPPORTED, std::string("device ") + prop.name + " is not sm_100a; this library is built for B200 only"));
  s->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess)
    return bail(fail(OCP_B200_ERR_CUDA, "cudaStreamCreate failed"));
  int rc = upload_pattern(s, d->num_blocks, d->block_ptr);
  if (rc != OCP_B200_OK) return bail(rc);
  rc = plan_launch(s);
  if (rc != OCP_B200_OK) return bail(rc);
  if (d->model_library && d->model_library[0]) {
    rc = load_model(s, d->model_library);
    if (rc != OCP_B200_OK) return bail(rc);
  }
  *out = s;
  return OCP_B200_OK;
}

int ocp_b200_destroy(ocp_b200_solver* s) {
  if (!s) return OCP_B200_OK;
  DeviceGuard device_guard_;
  device_guard_.enter(s->device);
  if (s->stream) { cudaStreamSynchronize(s->stream); cudaStreamDestroy(s->stream); }
  s->d_idx.release(); s->d_int.release(); s->d_kent.release(); s->d_krun.release(); s->d_arena.release();
  DevBuf<double>* bufs[] = {&s->hv, &s->q, &s->av, &s->l, &s->u, &s->solx, &s->soly, &s->info, &s->slab, &s->trace,
                            &s->x, &s->p, &s->frames, &s->lbx, &s->ubx, &s->lbg, &s->ubg, &s->f, &s->stats};
  for (DevBuf<double>* b : bufs) b->release();
  s->counter.release();
  s->phase.release();
  // the stage library stays loaded: its kernels are registered with the CUDA runtime and
  // unloading a module that another handle still uses would invalidate them
  delete s;
  return OCP_B200_OK;
}

int ocp_b200_update_settings(ocp_b200_solver* s, const ocp_b200_settings* settings) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  RC_TRY(check_settings(settings));
  const int old = s->settings.pcg_precond;
  s->settings = *settings;
  if (old != settings->pcg_precond) {
    ENTER_DEVICE(s->device);
    RC_TRY(plan_launch(s));
  }
  return OCP_B200_OK;
}

int ocp_b200_get_settings(const ocp_b200_solver* s, ocp_b200_settings* out) {
  if (!s || !out) return fail(OCP_B200_ERR_INVALID, "solver/out is NULL");
  *out = s->settings;
  return OCP_B200_OK;
}

int ocp_b200_solve_batch_device(ocp_b200_solver* s, int B, const double* d_frames, const double* d_p,
                                const double* d_lbx, const double* d_ubx, const double* d_lbg,
                                const double* d_ubg, double* d_x, double* d_f, double* d_stats, void* stream) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (B < 0 || (B > 0 && (!d_x || (s->np > 0 && !d_p) || !d_lbx || !d_ubx || (s->ng > 0 && (!d_lbg || !d_ubg)))))
    return fail(OCP_B200_ERR_INVALID, "bad arguments to solve_batch");
  if (B == 0) return OCP_B200_OK;
  if (!s->assemble) return fail(OCP_B200_ERR_MODEL, "this handle has no stage library (QP-only handle)");
  ENTER_DEVICE(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RC_TRY(reserve_qp(s, B));
  CUDA_TRY(s->stats.reserve(size_t(B) * OCP_B200_NSTATS));
  CUDA_TRY(s->f.reserve(B));
  double* stats = d_stats ? d_stats : s->stats.p;
  double* f = d_f ? d_f : s->f.p;
  if (s->settings.sqp_step_num == 0)
    CUDA_TRY(cudaMemsetAsync(stats, 0, size_t(B) * OCP_B200_NSTATS * sizeof(double), st));
  for (int step = 0; step < s->settings.sqp_step_num; ++step) {
    RC_TRY(assemble_on(s, B, d_x, d_p, d_frames, d_lbx, d_ubx, d_lbg, d_ubg, st));
    SolveArgs A{};
    A.B = B;
    A.h_vals = s->hv.p; A.ld_h = s->nnz_h; A.q = s->q.p; A.ld_n = s->n; A.a_vals = s->av.p; A.ld_a = s->nnz_a;
    A.l = s->l.p; A.u = s->u.p; A.ld_m = s->m;
    A.x_iter = d_x; A.np = s->np; A.N = s->N; A.sqp_alpha = s->settings.sqp_alpha;
    A.stats = stats; A.first_step = step == 0;
    RC_TRY(launch_admm(s, A, st));
  }
  {
    ProfScope prof(s, OCP_B200_PROF_OBJECTIVE, st);
    const int rc = s->objective(B, d_x, d_p, f, st);
    if (rc != 0) return fail(OCP_B200_ERR_CUDA, std::string("objective launch: ") + cudaGetErrorString(static_cast<cudaError_t>(rc)));
    s->launches++;
    ocpb200::store_objective_kernel<<<(B + 255) / 256, 256, 0, st>>>(B, f, stats);
    CUDA_TRY(cudaGetLastError());
    s->launches++;
  }
  return OCP_B200_OK;
}

int ocp_b200_shift_iterate_device(ocp_b200_solver* s, int B, double* d_x, void* stream) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (B < 0 || (B > 0 && !d_x)) return fail(OCP_B200_ERR_INVALID, "bad arguments to shift_iterate");
  if (B == 0 || s->N <= s->nf) return OCP_B200_OK;
  const size_t smem = size_t(s->N) * sizeof(double);
  if (smem > 48 * 1024) return fail(OCP_B200_ERR_UNSUPPORTED, "shift_iterate: trajectory longer than 6144 values");
  ENTER_DEVICE(s->device);
  ocpb200::shift_iterate_kernel<<<B, 256, smem, static_cast<cudaStream_t>(stream)>>>(s->nf, s->N, d_x);
  CUDA_TRY(cudaGetLastError());
  s->launches++;
  return OCP_B200_OK;
}

int ocp_b200_solve_batch(ocp_b200_solver* s, int B, const double* frames, const double* p, const double* lbx,
                         const double* ubx, const double* lbg, const double* ubg, double* x_inout, double* f_out,
                         double* stats) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (B < 0 || (B > 0 && (!x_inout || (s->np > 0 && !p) || !lbx || !ubx || (s->ng > 0 && (!lbg || !ubg)))))
    return fail(OCP_B200_ERR_INVALID, "bad arguments to solve_batch");
  if (B == 0) return OCP_B200_OK;
  ENTER_DEVICE(s->device);
  cudaStream_t st = s->stream;
  RC_TRY(upload_problem_inputs(s, B, frames, p, lbx, ubx, lbg, ubg, st));
  CUDA_TRY(s->x.reserve(size_t(B) * s->N));
  CUDA_TRY(s->f.reserve(B));
  CUDA_TRY(s->stats.reserve(size_t(B) * OCP_B200_NSTATS));
  RC_TRY(h2d(s->x.p, x_inout, size_t(B) * s->N, st));
  RC_TRY(ocp_b200_solve_batch_device(s, B, frames ? s->frames.p : nullptr, s->p.p, s->lbx.p, s->ubx.p, s->lbg.p,
                                     s->ubg.p, s->x.p, s->f.p, s->stats.p, st));
  RC_TRY(d2h(x_inout, s->x.p, size_t(B) * s->N, st));
  if (f_out) RC_TRY(d2h(f_out, s->f.p, B, st));
  if (stats) RC_TRY(d2h(stats, s->stats.p, size_t(B) * OCP_B200_NSTATS, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return OCP_B200_OK;
}

int ocp_b200_export_qp(ocp_b200_solver* s, int B, const double* frames, const double* p, const double* lbx,
                       const double* ubx, const double* lbg, const double* ubg, const double* x, double* h_vals,
                       double* q, double* a_vals, double* l, double* u) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (B <= 0 || !x || (s->np > 0 && !p) || !lbx || !ubx || (s->ng > 0 && (!lbg || !ubg)))
    return fail(OCP_B200_ERR_INVALID, "bad arguments to export_qp");
  ENTER_DEVICE(s->device);
  cudaStream_t st = s->stream;
  RC_TRY(upload_problem_inputs(s, B, frames, p, lbx, ubx, lbg, ubg, st));
  CUDA_TRY(s->x.reserve(size_t(B) * s->N));
  RC_TRY(h2d(s->x.p, x, size_t(B) * s->N, st));
  RC_TRY(reserve_qp(s, B));
  RC_TRY(assemble_on(s, B, s->x.p, s->p.p, frames ? s->frames.p : nullptr, s->lbx.p, s->ubx.p, s->lbg.p, s->ubg.p, st));
  if (h_vals) RC_TRY(d2h(h_vals, s->hv.p, size_t(B) * s->nnz_h, st));
  if (q) RC_TRY(d2h(q, s->q.p, size_t(B) * s->n, st));
  if (a_vals) RC_TRY(d2h(a_vals, s->av.p, size_t(B) * s->nnz_a, st));
  if (l) RC_TRY(d2h(l, s->l.p, size_t(B) * s->m, st));
  if (u) RC_TRY(d2h(u, s->u.p, size_t(B) * s->m, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return OCP_B200_OK;
}

static int qp_solve_common(ocp_b200_solver* s, int B, const double* h_vals, const double* q, const double* a_vals,
                           const double* l, const double* u, double* x_out, double* y_out, double* info,
                           int max_records, double* trace, int* n_records) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (B <= 0 || (s->nnz_h > 0 && !h_vals) || !q || !a_vals || !l || !u)
    return fail(OCP_B200_ERR_INVALID, "bad arguments to qp_solve");
  ENTER_DEVICE(s->device);
  cudaStream_t st = s->stream;
  RC_TRY(reserve_qp(s, B));
  CUDA_TRY(s->solx.reserve(size_t(B) * s->n));
  CUDA_TRY(s->soly.reserve(size_t(B) * s->m));
  CUDA_TRY(s->info.reserve(size_t(B) * OCP_B200_NINFO));
  RC_TRY(h2d(s->hv.p, h_vals, size_t(B) * s->nnz_h, st));
  RC_TRY(h2d(s->q.p, q, size_t(B) * s->n, st));
  RC_TRY(h2d(s->av.p, a_vals, size_t(B) * s->nnz_a, st));
  RC_TRY(h2d(s->l.p, l, size_t(B) * s->m, st));
  RC_TRY(h2d(s->u.p, u, size_t(B) * s->m, st));
  SolveArgs A{};
  A.B = B;
  A.h_vals = s->hv.p; A.ld_h = s->nnz_h; A.q = s->q.p; A.ld_n = s->n; A.a_vals = s->av.p; A.ld_a = s->nnz_a;
  A.l = s->l.p; A.u = s->u.p; A.ld_m = s->m;
  A.sol_x = s->solx.p; A.sol_y = s->soly.p; A.info = s->info.p;
  DevBuf<int> ntr;
  if (trace && max_records > 0) {
    CUDA_TRY(s->trace.reserve(size_t(max_records) * OCP_B200_TRACE_WIDTH));
    CUDA_TRY(ntr.reserve(1));
    CUDA_TRY(cudaMemsetAsync(ntr.p, 0, sizeof(int), st));
    A.trace = s->trace.p; A.max_trace = max_records; A.n_trace = ntr.p;
  }
  int rc = launch_admm(s, A, st);
  if (rc == OCP_B200_OK && x_out) rc = d2h(x_out, s->solx.p, size_t(B) * s->n, st);
  if (rc == OCP_B200_OK && y_out) rc = d2h(y_out, s->soly.p, size_t(B) * s->m, st);
  if (rc == OCP_B200_OK && info) rc = d2h(info, s->info.p, size_t(B) * OCP_B200_NINFO, st);
  int nrec = 0;
  if (rc == OCP_B200_OK && A.trace) {
    cudaError_t e = cudaMemcpyAsync(&nrec, ntr.p, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail(OCP_B200_ERR_CUDA, cudaGetErrorString(e));
    else rc = d2h(trace, s->trace.p, size_t(std::min(nrec, max_records)) * OCP_B200_TRACE_WIDTH, st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  ntr.release();
  if (rc != OCP_B200_OK) return rc;
  if (e != cudaSuccess) return fail(OCP_B200_ERR_CUDA, std::string("qp_solve: ") + cudaGetErrorString(e));
  if (n_records) *n_records = std::min(nrec, max_records);
  return OCP_B200_OK;
}

int ocp_b200_qp_solve_batch(ocp_b200_solver* s, int B, const double* h_vals, const double* q, const double* a_vals,
                            const double* l, const double* u, double* x_out, double* y_out, double* info) {
  return qp_solve_common(s, B, h_vals, q, a_vals, l, u, x_out, y_out, info, 0, nullptr, nullptr);
}

int ocp_b200_admm_trace(ocp_b200_solver* s, const double* h_vals, const double* q, const double* a_vals,
                        const double* l, const double* u, int max_records, double* trace, int* n_records,
                        double* x_out, double* y_out) {
  if (!trace || max_records <= 0 || !n_records) return fail(OCP_B200_ERR_INVALID, "trace buffer missing");
  return qp_solve_common(s, 1, h_vals, q, a_vals, l, u, x_out, y_out, nullptr, max_records, trace, n_records);
}

long long ocp_b200_launch_count(const ocp_b200_solver* s) { return s ? s->launches : 0; }

int ocp_b200_set_profiling(ocp_b200_solver* s, int enabled) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  s->profiling = enabled < 0 ? 0 : (enabled > 2 ? 2 : enabled);
  if (enabled >= 2) {
    ENTER_DEVICE(s->device);
    CUDA_TRY(s->phase.reserve(OCP_B200_NPHASE));
    CUDA_TRY(cudaMemset(s->phase.p, 0, OCP_B200_NPHASE * sizeof(long long)));
  }
  return OCP_B200_OK;
}

int ocp_b200_get_phase_cycles(ocp_b200_solver* s, long long* cycles) {
  if (!s || !cycles) return fail(OCP_B200_ERR_INVALID, "solver/cycles is NULL");
  if (!s->phase.p) { for (int k = 0; k < OCP_B200_NPHASE; ++k) cycles[k] = 0; return OCP_B200_OK; }
  ENTER_DEVICE(s->device);
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(cycles, s->phase.p, OCP_B200_NPHASE * sizeof(long long), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemset(s->phase.p, 0, OCP_B200_NPHASE * sizeof(long long)));
  return OCP_B200_OK;
}

int ocp_b200_get_profile(ocp_b200_solver* s, double* ms, long long* count, int reset) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  ENTER_DEVICE(s->device);
  for (size_t k = 0; k < s->ev_kind.size(); ++k) {
    cudaEvent_t a = s->ev[2 * k], b = s->ev[2 * k + 1];
    CUDA_TRY(cudaEventSynchronize(b));
    float t = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&t, a, b));
    s->prof_ms[s->ev_kind[k]] += t;
    s->prof_count[s->ev_kind[k]]++;
    cudaEventDestroy(a); cudaEventDestroy(b);
  }
  s->ev.clear(); s->ev_kind.clear();
  for (int k = 0; k < OCP_B200_NPROF; ++k) {
    if (ms) ms[k] = s->prof_ms[k];
    if (count) count[k] = s->prof_count[k];
    if (reset) { s->prof_ms[k] = 0; s->prof_count[k] = 0; }
  }
  return OCP_B200_OK;
}

int ocp_b200_get_dims(const ocp_b200_solver* s, int* n, int* m, int* nnz_h, int* nnz_a, int* smem_bytes,
                      int* resident) {
  if (!s) return fail(OCP_B200_ERR_INVALID, "solver is NULL");
  if (n) *n = s->n;
  if (m) *m = s->m;
  if (nnz_h) *nnz_h = s->nnz_h;
  if (nnz_a) *nnz_a = s->nnz_a;
  if (smem_bytes) *smem_bytes = s->wide.smem_bytes;
  // PCG kernel: bit 0 = its state is in shared memory.  Direct kernels: bit 0 = the latency plan keeps everything in
  // shared memory, bit 1 set, bits 2 and up = placement of the throughput plan.
  if (resident)
    *resident = s->wide.place < 0 ? s->wide.smem_bytes > 0 : (s->deep.place == 1) | 2 | s->wide.place << 2;
  return OCP_B200_OK;
}

// ---- several devices from one process ------------------------------------------------------------------------
struct ocp_b200_multi {
  std::vector<ocp_b200_solver*> handles;
  std::vector<int> devices;
  int np = 0, nf = 0, N = 0;
};

int ocp_b200_multi_partition(int B, int ndev, int* offsets) {
  if (B < 0 || ndev <= 0 || !offsets) return fail(OCP_B200_ERR_INVALID, "bad arguments to multi_partition");
  const int per = (B + ndev - 1) / ndev;   // contiguous blocks of ceil(B / ndev), the tail devices may get less / nothing
  for (int k = 0; k <= ndev; ++k) offsets[k] = std::min(B, k * per);
  return OCP_B200_OK;
}

int ocp_b200_create_multi(const ocp_b200_problem_desc* desc, const ocp_b200_settings* settings, const int* devices,
                          int ndev, ocp_b200_multi** out) {
  if (!desc || !out || !devices || ndev <= 0) return fail(OCP_B200_ERR_INVALID, "bad arguments to create_multi");
  *out = nullptr;
  ocp_b200_multi* m = new (std::nothrow) ocp_b200_multi();
  if (!m) return fail(OCP_B200_ERR_INVALID, "out of host memory");
  for (int k = 0; k < ndev; ++k) {
    ocp_b200_problem_desc d = *desc;
    d.device = devices[k];
    ocp_b200_solver* h = nullptr;
    const int rc = ocp_b200_create(&d, settings, &h);
    if (rc != OCP_B200_OK) {
      const std::string keep = g_error;
      ocp_b200_destroy_multi(m);
      return fail(rc, "device " + std::to_string(devices[k]) + ": " + keep);
    }
    m->handles.push_back(h);
    m->devices.push_back(devices[k]);
  }
  m->np = desc->np; m->nf = desc->nf; m->N = desc->nf * desc->horizon;
  *out = m;
  return OCP_B200_OK;
}

int ocp_b200_destroy_multi(ocp_b200_multi* m) {
  if (!m) return OCP_B200_OK;
  for (ocp_b200_solver* h : m->handles) ocp_b200_destroy(h);
  delete m;
  return OCP_B200_OK;
}

int ocp_b200_multi_update_settings(ocp_b200_multi* m, const ocp_b200_settings* settings) {
  if (!m) return fail(OCP_B200_ERR_INVALID, "multi handle is NULL");
  for (ocp_b200_solver* h : m->handles) RC_TRY(ocp_b200_update_settings(h, settings));
  return OCP_B200_OK;
}

int ocp_b200_multi_device_count(const ocp_b200_multi* m) { return m ? static_cast<int>(m->handles.size()) : 0; }
ocp_b200_solver* ocp_b200_multi_handle(ocp_b200_multi* m, int k) {
  return (m && k >= 0 && k < static_cast<int>(m->handles.size())) ? m->handles[k] : nullptr;
}

int ocp_b200_solve_batch_multi(ocp_b200_multi* m, int B, const double* frames, const double* p, const double* lbx,
                               const double* ubx, const double* lbg, const double* ubg, double* x_inout,
                               double* f_out, double* stats) {
  if (!m || m->handles.empty()) return fail(OCP_B200_ERR_INVALID, "multi handle is NULL");
  if (B < 0) return fail(OCP_B200_ERR_INVALID, "bad arguments to solve_batch_multi");
  if (B == 0) return OCP_B200_OK;
  const int ndev = static_cast<int>(m->handles.size());
  std::vector<int> off(ndev + 1);
  RC_TRY(ocp_b200_multi_partition(B, ndev, off.data()));
  std::vector<int> rc(ndev, OCP_B200_OK);
  std::vector<std::string> err(ndev);
  auto work = [&](int k) {
    const int b0 = off[k], nb = off[k + 1] - off[k];
    if (nb <= 0) return;
    rc[k] = ocp_b200_solve_batch(m->handles[k], nb, frames ? frames + size_t(b0) * m->nf : nullptr,
                                 p ? p + size_t(b0) * m->np : nullptr, lbx, ubx, lbg, ubg,
                                 x_inout ? x_inout + size_t(b0) * m->N : nullptr, f_out ? f_out + b0 : nullptr,
                                 stats ? stats + size_t(b0) * OCP_B200_NSTATS : nullptr);
    if (rc[k] != OCP_B200_OK) err[k] = g_error;   // g_error is per thread
  };
  // one host thread per device: every ocp_b200_solve_batch uploads, launches, downloads and waits on its own stream
  std::vector<std::thread> threads;
  for (int k = 1; k < ndev; ++k) threads.emplace_back(work, k);
  work(0);
  for (std::thread& t : threads) t.join();
  for (int k = 0; k < ndev; ++k)
    if (rc[k] != OCP_B200_OK) return fail(rc[k], "device " + std::to_string(m->devices[k]) + ": " + err[k]);
  return OCP_B200_OK;
}

/* Test hook (not part of include/ocp_b200.h): compresses the CSC structure (ptr[nout + 1], val[nnz], optional
 * val2[nnz]) with periodic_index.h, expands it again and returns the number of 32-bit words of the compressed
 * form, or -1 when the structure cannot be represented / the expansion differs.  Pure host code. */
int ocp_b200_internal_compress_index(int nout, const int* ptr, const int* val, const int* val2, int* regions) {
  if (nout < 0 || !ptr || (!val && ptr[nout] > 0)) return -1;
  std::vector<int> p(ptr, ptr + nout + 1), v(val, val + ptr[nout]), v2;
  if (val2) v2.assign(val2, val2 + ptr[nout]);
  std::vector<int> periods;
  for (int q = 1; q <= 96; ++q) periods.push_back(q);
  ocpb200::PIndexHost h;
  if (!ocpb200::build_periodic_index(p, v, v2, periods, h)) return -1;
  if (regions) *regions = static_cast<int>(h.reg.size());
  return static_cast<int>(h.words());
}

int ocp_b200_get_plan(const ocp_b200_solver* s, int* v, int count) {
  if (!s || !v || count < 0) return fail(OCP_B200_ERR_INVALID, "solver/v is NULL");
  int o[OCP_B200_PLAN_COUNT] = {0};
  const int sms = std::max(1, s->num_sms);
  const LaunchPlan* L[2] = {&s->wide, &s->deep};
  for (int k = 0; k < 2; ++k) {
    o[5 * k + 0] = L[k]->place; o[5 * k + 1] = L[k]->threads; o[5 * k + 2] = L[k]->smem_bytes;
    o[5 * k + 3] = L[k]->max_ctas / sms; o[5 * k + 4] = static_cast<int>(L[k]->slab_doubles * sizeof(double) / 1024);
  }
  o[OCP_B200_PLAN_TRI_OK] = s->wide.place >= 0;
  o[OCP_B200_PLAN_TRI_NP] = s->pat.tri_np; o[OCP_B200_PLAN_TRI_BS] = s->pat.tri_bs; o[OCP_B200_PLAN_TRI_NB] = s->pat.tri_nb;
  o[OCP_B200_PLAN_NNZ_P] = s->nnz_p;
  o[OCP_B200_PLAN_NUM_SMS] = s->num_sms;
  for (int k = 0; k < count && k < OCP_B200_PLAN_COUNT; ++k) v[k] = o[k];
  return OCP_B200_OK;
}

}  // extern "C"
