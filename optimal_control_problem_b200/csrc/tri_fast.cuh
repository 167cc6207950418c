// tri_fast.cuh -- exact-size (compile-time BS) building blocks of the bordered block-tridiagonal
// LDL' of admm_direct_kernel.cuh: dot products, the one-warp block inverse, one sweep stage.
// tri_twisted.cuh assembles them into the factorisation and the solve.
//
// The sequential parts of the algorithm (the two sweeps of a solve, the Gauss-Jordan inverse
// of a diagonal block) run in ONE warp while the rest of the CTA waits, so what limits them is
// the length of that warp's instruction stream and its dependent-latency chain -- not memory
// bandwidth.  These versions therefore: unroll everything over BS with no predication, read
// block rows with 16-byte shared-memory loads (row pitch ld is even), split every block row
// over LPR = 32 / BS lanes (BS = 16: two lanes per row, one shuffle to combine), keep the next
// stage's block row in registers while the current one is multiplied, and hold one matrix
// column per lane in registers during the inverse.  No integer division in per-stage loops.
#pragma once

namespace ocpb200 {
namespace direct {

template <int BS> struct TriCfg {
  static constexpr int LPR = BS <= 8 ? 4 : (BS <= 16 ? 2 : 1);   // lanes per block row in the sweeps
  static constexpr int CPL = BS / LPR;                           // columns per lane
  static_assert(BS % LPR == 0 && CPL % 2 == 0, "block size must split into even lane chunks");
};

// sum_t a[t] * b[t],  both contiguous and 16-byte aligned, t < BS
template <int BS>
__device__ __forceinline__ double dot_cc(const double* __restrict__ a, const double* __restrict__ b) {
  const double2* a2 = reinterpret_cast<const double2*>(a);
  const double2* b2 = reinterpret_cast<const double2*>(b);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
  for (int t = 0; t < BS / 2; t += 2) {
    const double2 x0 = a2[t], y0 = b2[t];
    s0 = fma(x0.x, y0.x, s0); s1 = fma(x0.y, y0.y, s1);
    if (t + 1 < BS / 2) {
      const double2 x1 = a2[t + 1], y1 = b2[t + 1];
      s2 = fma(x1.x, y1.x, s2); s3 = fma(x1.y, y1.y, s3);
    }
  }
  return (s0 + s1) + (s2 + s3);
}

// sum_t a[t] * b[t * sb],  a contiguous and 16-byte aligned, b strided
template <int BS>
__device__ __forceinline__ double dot_cs(const double* __restrict__ a, const double* __restrict__ b, int sb) {
  const double2* a2 = reinterpret_cast<const double2*>(a);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
  for (int t = 0; t < BS / 2; t += 2) {
    const double2 x0 = a2[t];
    s0 = fma(x0.x, b[(2 * t) * sb], s0); s1 = fma(x0.y, b[(2 * t + 1) * sb], s1);
    if (t + 1 < BS / 2) {
      const double2 x1 = a2[t + 1];
      s2 = fma(x1.x, b[(2 * t + 2) * sb], s2); s3 = fma(x1.y, b[(2 * t + 3) * sb], s3);
    }
  }
  return (s0 + s1) + (s2 + s3);
}

// 2 x 2 tiles of the dot products above: o[2 i + j] = sum_t a_i[t] * b_j[t], every product and every partial sum
// exactly as in dot_cc / dot_cs (element t goes to accumulator t % 4, result (s0 + s1) + (s2 + s3)), but the four
// operands rows are loaded once for four results: a third of the shared-memory loads of four separate calls.
template <int BS>
__device__ __forceinline__ void tile_cc(const double* __restrict__ a0, const double* __restrict__ a1,
                                        const double* __restrict__ b0, const double* __restrict__ b1, double (&o)[4]) {
  const double2* A0 = reinterpret_cast<const double2*>(a0);
  const double2* A1 = reinterpret_cast<const double2*>(a1);
  const double2* B0 = reinterpret_cast<const double2*>(b0);
  const double2* B1 = reinterpret_cast<const double2*>(b1);
  double s[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { s[i][0] = 0.0; s[i][1] = 0.0; s[i][2] = 0.0; s[i][3] = 0.0; }
#pragma unroll 2
  for (int t = 0; t < BS / 2; ++t) {
    const double2 x0 = A0[t], x1 = A1[t], y0 = B0[t], y1 = B1[t];
    const int k = (t & 1) * 2;   // double2 t holds elements 2t, 2t + 1 -> accumulators (2t) % 4, (2t + 1) % 4
    s[0][k] = fma(x0.x, y0.x, s[0][k]); s[0][k + 1] = fma(x0.y, y0.y, s[0][k + 1]);
    s[1][k] = fma(x0.x, y1.x, s[1][k]); s[1][k + 1] = fma(x0.y, y1.y, s[1][k + 1]);
    s[2][k] = fma(x1.x, y0.x, s[2][k]); s[2][k + 1] = fma(x1.y, y0.y, s[2][k + 1]);
    s[3][k] = fma(x1.x, y1.x, s[3][k]); s[3][k + 1] = fma(x1.y, y1.y, s[3][k + 1]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = (s[i][0] + s[i][1]) + (s[i][2] + s[i][3]);
}
// a_i contiguous rows, b_j = two adjacent columns of a pitch-sb matrix starting at bcol (16-byte aligned)
template <int BS>
__device__ __forceinline__ void tile_cs(const double* __restrict__ a0, const double* __restrict__ a1,
                                        const double* __restrict__ bcol, int sb, double (&o)[4]) {
  const double2* A0 = reinterpret_cast<const double2*>(a0);
  const double2* A1 = reinterpret_cast<const double2*>(a1);
  double s[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { s[i][0] = 0.0; s[i][1] = 0.0; s[i][2] = 0.0; s[i][3] = 0.0; }
#pragma unroll 2
  for (int t = 0; t < BS / 2; ++t) {
    const double2 x0 = A0[t], x1 = A1[t];
    const double2 ya = *reinterpret_cast<const double2*>(bcol + (2 * t) * sb);       // row 2t:     columns j = 0, 1
    const double2 yb = *reinterpret_cast<const double2*>(bcol + (2 * t + 1) * sb);   // row 2t + 1
    const int k = (t & 1) * 2;
    s[0][k] = fma(x0.x, ya.x, s[0][k]); s[0][k + 1] = fma(x0.y, yb.x, s[0][k + 1]);
    s[1][k] = fma(x0.x, ya.y, s[1][k]); s[1][k + 1] = fma(x0.y, yb.y, s[1][k + 1]);
    s[2][k] = fma(x1.x, ya.x, s[2][k]); s[2][k + 1] = fma(x1.y, yb.x, s[2][k + 1]);
    s[3][k] = fma(x1.x, ya.y, s[3][k]); s[3][k + 1] = fma(x1.y, yb.y, s[3][k + 1]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = (s[i][0] + s[i][1]) + (s[i][2] + s[i][3]);
}

// in-place inverse of an SPD BS x BS block (Gauss-Jordan, no pivoting) by ONE warp.
// Lane c < BS holds column c in registers.  Per pivot k the multipliers f[r] = -M[r][k] / M[k][k]
// are needed by every lane; M[r][k] is (up to the sign flip of already pivoted rows) element k of
// lane r's own column, because the working matrix stays symmetric among unpivoted indices:
// lane k broadcasts 1 / M[k][k] (one shuffle), every lane forms its own f[r] with one multiply and
// the 16 values are all-gathered through `piv` (16-byte aligned scratch of >= BS doubles).  The
// serial part of a pivot is reciprocal -> shuffle -> multiply -> store/load round trip -> FMAs.
// kStoreT: the inverse is stored column-major with pitch BS (element (r, c) at M[c * BS + r]) in the first BS * BS
// doubles of the block; the input is read row-major with pitch LD as always.
template <int BS, int LD = BS + 2, bool kStoreT = false>
__device__ __forceinline__ void warp_invert_exact(double* M, int /*ld*/, int lane, double* piv) {
  constexpr int ld = LD;
  static_assert(BS % 2 == 0 && BS <= 32, "one column per lane, even size");
  const bool act = lane < BS;
  const int cc = act ? lane : 0;
  double col[BS];
#pragma unroll
  for (int r = 0; r < BS; ++r) col[r] = M[r * ld + cc];
  const double2* piv2 = reinterpret_cast<const double2*>(piv);
  // 1 / M[k][k] of the NEXT pivot is started by its owner (lane k + 1) as soon as this pivot's multiplier is known:
  // M[k+1][k+1] <- fma(f[k+1], M[k][k+1], M[k+1][k+1]) is the very update the loop below applies to that element, so
  // the bits are the same, but the reciprocal (~80 cycles) now overlaps the all-gather round trip and the FMAs
  // instead of heading the next pivot's dependency chain
  double rnext = 1.0 / col[0];   // lane 0: 1 / M[0][0]
#pragma unroll
  for (int k = 0; k < BS; ++k) {
    const double ck = col[k];                                   // M[k][c] == M[c][k]
    const double ipiv = __shfl_sync(0xffffffffu, rnext, k);     // every lane: 1 / M[k][k]
    const bool mine = lane == k;
    // f[lane] = -M[lane][k] / M[k][k].  Rows already pivoted hold the sign-flipped coupling
    // (M[r][k] == -M[k][r] for r < k in in-place Gauss-Jordan), rows still to come are symmetric.
    const double fl = mine ? ipiv : (lane < k ? ck * ipiv : -ck * ipiv);
    if (act) piv[lane] = fl;
    if (k + 1 < BS) rnext = 1.0 / fma(fl, ck, col[k + 1 < BS ? k + 1 : k]);   // meaningful on lane k + 1 only
    __syncwarp();
#pragma unroll
    for (int r = 0; r < BS / 2; ++r) {
      const double2 f = piv2[r];
      const int r0 = 2 * r, r1 = 2 * r + 1;
      col[r0] = mine ? f.x : (r0 == k ? ck * f.x : fma(f.x, ck, col[r0]));
      col[r1] = mine ? f.y : (r1 == k ? ck * f.y : fma(f.y, ck, col[r1]));
    }
    __syncwarp();
  }
  if (act) {
    if constexpr (kStoreT) {   // (every lane read its column before the first __syncwarp above: in place is safe)
      double2* out = reinterpret_cast<double2*>(M + lane * BS);
#pragma unroll
      for (int r = 0; r < BS / 2; ++r) out[r] = make_double2(col[2 * r], col[2 * r + 1]);
    } else {
#pragma unroll
      for (int r = 0; r < BS; ++r) M[r * ld + lane] = col[r];
    }
  }
}

// D_p^-1 (np x np, pitch np + 1): exact-size code for the border sizes of the benchmark problems
__device__ __forceinline__ void invert_border(double* Dp, int np, int lane, double* piv) {
  if (np == 12) warp_invert_exact<12, 13>(Dp, 13, lane, piv);
  else if (np == 4) warp_invert_exact<4, 5>(Dp, 5, lane, piv);
  else if (np == 24) warp_invert_exact<24, 25>(Dp, 25, lane, piv);
  else warp_invert(Dp, np, np + 1, lane);
}

// one stage of a sweep: dst[r] -= sum_c Lpart[c] * src[c] over this lane's CPL columns, combined
// over the LPR lanes of the row
template <int BS>
__device__ __forceinline__ void sweep_stage(const double (&Lpart)[TriCfg<BS>::CPL], const double* __restrict__ src,
                                            double* __restrict__ dst, bool writer) {
  constexpr int CPL = TriCfg<BS>::CPL, LPR = TriCfg<BS>::LPR;
  const double old = writer ? *dst : 0.0;   // issued before the chain, not after the shuffle
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
  for (int c = 0; c < CPL; c += 4) {
    s0 = fma(Lpart[c], src[c], s0);
    s1 = fma(Lpart[c + 1], src[c + 1], s1);
    if (c + 2 < CPL) { s2 = fma(Lpart[c + 2], src[c + 2], s2); s3 = fma(Lpart[c + 3], src[c + 3], s3); }
  }
  double s = (s0 + s1) + (s2 + s3);
  if (LPR >= 2) s += __shfl_xor_sync(0xffffffffu, s, 1);
  if (LPR >= 4) s += __shfl_xor_sync(0xffffffffu, s, 2);
  if (writer) *dst = old - s;
  __syncwarp();
}

}  // namespace direct
}  // namespace ocpb200
