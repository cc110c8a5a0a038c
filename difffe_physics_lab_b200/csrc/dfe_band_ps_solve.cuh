// Both banded triangular sweeps of one per-sample factor by one warp: L y = b, then L^T x = y.  k_bps_solve (dfe_band_ps.cu)
// and k_hps_roll (dfe_heat.cu) call it.  Included inside an anonymous namespace, after dfe_internal.h.
//
// The factor is one sample's slice of k_bps_factor's output: invd[npad] | Lr[npad * 32] with invd[i] = 1 / L_ii and
// Lr[i * 32 + d - 1] = L[i][i - d].  Lane a owns row 32k + a of block row k.  Per block row: the coupling to the previous
// (next) block row, 32 fmas per lane with the neighbour's solution broadcast by shuffles, then the 32 dependent steps of the
// triangular diagonal block.  One read of L per sweep.
//
//   rhs(i)      entry i of b; called by the lane that owns row i, before that lane writes x[i]
//   out(i, xv)  entry i of the solution x; the lane that owns row i
// y stays in x (npad doubles) between the sweeps: the lane that wrote an entry reads it back, so no synchronisation.
#pragma once

template <class Rhs, class Out>
__device__ __forceinline__ void bps_sweeps(const double* __restrict__ invd, const double* __restrict__ Lr, double* x, int nb,
                                           int lane, Rhs rhs, Out out) {
  constexpr unsigned full = 0xffffffffu;
  double prev = 0.0;   // lane c: entry c of the solution of the block row just finished
  for (int k = 0; k < nb; ++k) {
    const int i = 32 * k + lane;
    const double* Li = Lr + static_cast<size_t>(i) * 32;   // Li[d - 1] = L[i][i - d]
    double acc = rhs(i);
    if (k > 0) {
#pragma unroll
      for (int c = 0; c < 32; ++c) {   // L[i][32(k-1) + c], d = 32 + lane - c
        const double yc = __shfl_sync(full, prev, c);
        if (c >= lane) acc = fma(-Li[31 + lane - c], yc, acc);
      }
    }
    const double inv = invd[i];
    double y = 0.0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {     // L[i][32k + j], d = lane - j
      const double yj = __shfl_sync(full, acc * inv, j);
      if (lane == j) y = yj;
      if (lane > j) acc = fma(-Li[lane - j - 1], yj, acc);
    }
    x[i] = y;
    prev = y;
  }
  prev = 0.0;
  for (int k = nb - 1; k >= 0; --k) {
    const int i = 32 * k + lane;
    double acc = x[i];
    if (k + 1 < nb) {
      const double* Ln = Lr + static_cast<size_t>(32 * (k + 1)) * 32;
#pragma unroll
      for (int c = 0; c < 32; ++c) {   // L[32(k+1) + c][i], d = 32 + c - lane
        const double xc = __shfl_sync(full, prev, c);
        if (c <= lane) acc = fma(-Ln[c * 32 + 31 + c - lane], xc, acc);
      }
    }
    const double inv = invd[i];
    const double* Lk = Lr + static_cast<size_t>(32 * k) * 32;
    double xv = 0.0;
#pragma unroll
    for (int j = 31; j >= 0; --j) {    // L[32k + j][i], d = j - lane
      const double xj = __shfl_sync(full, acc * inv, j);
      if (lane == j) xv = xj;
      if (lane < j) acc = fma(-Lk[j * 32 + (j - lane) - 1], xj, acc);
    }
    out(i, xv);
    prev = xv;
  }
}
