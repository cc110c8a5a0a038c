// The block-row step of the banded triangular solves on the FP64 tensor cores (DMMA m8n8k4) and the layout of its B-operand
// fragments: k_band_blocks (dfe_batch.cu) writes the fragments, k_band_solve_mma (dfe_batch.cu) and k_heat_roll
// (dfe_heat.cu) read them.  Included inside an anonymous namespace, after dfe_internal.h.
//
// With 32 x 32 blocks the band of L is block-bidiagonal: L y = b reads  y_k = H_k (b_k - S_k y_{k-1})  with H_k = L_kk^{-1}
// (lower triangular) and S_k = L_{k,k-1} (UPPER triangular: the band is 32 wide), and L^T x = y reads
// x_k = H_k^T (y_k - S_{k+1}^T x_{k+1}).  The solve works on the transposed problem (samples x rows),
// Y_k^T = (B_k^T - Y_{k-1}^T S_k^T) H_k^T, so that a warp's 16 samples are the M dimension (two 8-row tiles) and the previous
// block's result is the A operand of the next product.  The accumulator layout of m8n8k4 (thread t holds row t/4, columns
// 2(t%4), 2(t%4)+1 of an 8 x 8 tile) differs from the A layout (row t/4, column t%4) — but a contraction may enumerate its k
// index in any order as long as both operands agree: k-step (tile ntp, half j) is DEFINED to cover the columns
// 8ntp + 2(t%4) + j, which are exactly the accumulator registers the thread already holds.  The B fragments are stored with
// the matching permutation, and the result of one block row feeds the next one without a shuffle or shared-memory round trip.
#pragma once

constexpr int FRAGD = dfe::BAND_FRAGD;   // doubles per block row and direction: H fragments (1024), then -S fragments (1024)
constexpr int MMA_S = 16;                // samples per warp (two m8 tiles)

// 16 samples x 32 columns of one block row in the accumulator layout: [mt][nt][j] is sample 8 mt + lane / 4,
// column 8 nt + 2 (lane % 4) + j
typedef double Blk[2][4][2];

// B register of `lane` for k-step (ntp, j) and output tile nt: entry frag_idx(ntp, j, nt, lane) of a 1024-double half
__device__ __forceinline__ int frag_idx(int ntp, int j, int nt, int lane) { return ((ntp * 2 + j) * 4 + nt) * 32 + lane; }
// the inverse, for the writer: entry q of a half holds M[r][c] of the 32 x 32 block M (r: output column, c: k index)
__device__ __forceinline__ void frag_rc(int q, int& r, int& c) {
  const int f = q >> 5, t = q & 31;
  r = 8 * (f & 3) + (t >> 2);
  c = 8 * (f >> 3) + 2 * (t & 3) + ((f >> 2) & 1);
}

// the 2 nb steps of one solve: block rows 0 .. nb-1 (forward), then nb-1 .. 0 (backward); -1 past the end
__device__ __forceinline__ int band_block(int step, int nb) { return step < nb ? step : 2 * nb - 1 - step; }
__device__ __forceinline__ const double* frag_src(const double* Ff, const double* Bf, int nb, int step) {
  return step < nb ? Ff + static_cast<size_t>(step) * FRAGD : Bf + static_cast<size_t>(2 * nb - 1 - step) * FRAGD;
}

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ void blk_copy(Blk& d, const Blk& s) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      d[mt][nt][0] = s[mt][nt][0];
      d[mt][nt][1] = s[mt][nt][1];
    }
}
// block kb of two sample rows; row[mt] points at column 2 (lane % 4) of the row of sample mt (16-byte aligned)
__device__ __forceinline__ void ld_block(double* const (&row)[2], int kb, Blk& R) {
#pragma unroll
  for (int nt = 0; nt < 4; ++nt)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const double2 v = *reinterpret_cast<const double2*>(row[mt] + 32 * kb + 8 * nt);
      R[mt][nt][0] = v.x;
      R[mt][nt][1] = v.y;
    }
}

// Step `step` of the solve on block row k = band_block(step, nb), with that step's fragments staged at `stg`.  t holds the
// right-hand side of block k (overwritten), P the result of the previous step; acc receives the result of this one.
//   stage 1: t += P (-S_k)^T (forward) / P (-S_{k+1}) (backward); skipped on the first block row of a pass
//   stage 2: acc = t H_k^T (forward) / t H_k (backward)
// S and H are triangular: 10 of the 16 8 x 8 tiles of each are non-zero, and only those are multiplied.
__device__ __forceinline__ void band_step(int step, int nb, const double* stg, int lane, Blk& t, const Blk& P, Blk& acc) {
  const double* sH = stg;
  const double* sG = stg + 1024;
  if (step != 0 && step != nb) {
    if (step < nb) {
#pragma unroll
      for (int ntp = 0; ntp < 4; ++ntp)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int nt = 0; nt <= ntp; ++nt) {     // t[s][r] += y_prev[s][c] (-S[r][c]), zero for c < r
            const double b = sG[frag_idx(ntp, j, nt, lane)];
            dmma884(t[0][nt][0], t[0][nt][1], P[0][ntp][j], b);
            dmma884(t[1][nt][0], t[1][nt][1], P[1][ntp][j], b);
          }
    } else {
#pragma unroll
      for (int ntp = 0; ntp < 4; ++ntp)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int nt = ntp; nt < 4; ++nt) {      // t[s][r] += x_next[s][c] (-U[c][r]), zero for c > r
            const double b = sG[frag_idx(ntp, j, nt, lane)];
            dmma884(t[0][nt][0], t[0][nt][1], P[0][ntp][j], b);
            dmma884(t[1][nt][0], t[1][nt][1], P[1][ntp][j], b);
          }
    }
  }
  // the accumulators of stage 1 are the A operand of stage 2 (see the layout note above)
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
  if (step < nb) {
#pragma unroll
    for (int ntp = 0; ntp < 4; ++ntp)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int nt = ntp; nt < 4; ++nt) {        // out[s][r] += t[s][c] H[r][c], zero for c > r
          const double b = sH[frag_idx(ntp, j, nt, lane)];
          dmma884(acc[0][nt][0], acc[0][nt][1], t[0][ntp][j], b);
          dmma884(acc[1][nt][0], acc[1][nt][1], t[1][ntp][j], b);
        }
  } else {
#pragma unroll
    for (int ntp = 0; ntp < 4; ++ntp)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int nt = 0; nt <= ntp; ++nt) {       // out[s][r] += t[s][c] H[c][r], zero for c < r
          const double b = sH[frag_idx(ntp, j, nt, lane)];
          dmma884(acc[0][nt][0], acc[0][nt][1], t[0][ntp][j], b);
          dmma884(acc[1][nt][0], acc[1][nt][1], t[1][ntp][j], b);
        }
  }
}
