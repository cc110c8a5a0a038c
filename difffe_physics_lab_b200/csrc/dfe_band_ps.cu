// Batched banded direct solve when every sample has its own conductivity (kappa (B, 1) or (B, n_el)) on a 2-D P1 mesh
// whose K_free has half bandwidth <= 32 (dfe_band_supported).  The shared-kappa route (dfe_batch.cu) factors one matrix
// and runs the tensor-core block TRSM over the batch; here every sample has its own matrix, so the per-sample work is
//   assemble      k_bps_assemble   vals_full of sample b, (B, nnz_full): assemble_row (dfe_assemble_row.cuh), the
//                                  arithmetic of dfe_assemble, so each matrix is bit-identical to dfe_assemble(kappa_b)
//   factor        k_bps_factor     K_free(kappa_b) = L_b L_b^T, blocked: the per-entry operation order of
//                                  k_band_factor_blk, so each factor is bit-identical to dfe_band_factor on that matrix;
//                                  block rows are read straight from the sample's vals_full through the K_free pattern
//   load          k_band_rhs_fwd   (dfe_batch.cu) with a per-sample vals_full stride for the lifting
//   solve         k_bps_solve      L_b y = b, L_b^T x = y: one warp per sample, both sweeps, one read of L_b per sweep
//                                  (bps_sweeps, dfe_band_ps_solve.cuh, shared with the per-sample heat rollout)
//   gradients     k_band_grad2 / k_band_grad (dfe_batch.cu): they already write per-sample dL/dkappa and dL/df
// Every reduction has a fixed order (no float atomics): the results are bit-reproducible and independent of B.
#include "dfe_internal.h"

namespace {

using dfe::MeshDev;
#include "dfe_assemble_row.cuh"   // assemble_row: the per-sample matrices of dfe_assemble
#include "dfe_band_ps_solve.cuh"  // bps_sweeps: both banded sweeps of one sample's factor by one warp

constexpr int BW = 32;            // half bandwidth supported (as dfe_batch.cu)
constexpr int FT = 128;           // threads per CTA of the factor kernel (one CTA per sample)
constexpr int SW_ = 4;            // warps per CTA of the solve kernel (one warp per sample)
constexpr unsigned FULL = 0xffffffffu;

// vals_full of every sample: thread (p, b) assembles row p of sample b
__global__ void k_bps_assemble(const MeshDev M, long long B, const double* __restrict__ kappa, int per_elem,
                               double* __restrict__ vals) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_nodes) return;
  const bool local = M.rowptr[p + 1] - M.rowptr[p] <= ROWMAX;
  const long long kst = per_elem ? M.n_el : 1;
  for (long long b = blockIdx.y; b < B; b += gridDim.y) {
    double* vb = vals + b * M.nnz_full;
    if (local) assemble_row<true, false>(M, p, kappa + b * kst, per_elem, nullptr, vb, nullptr);
    else assemble_row<false, false>(M, p, kappa + b * kst, per_elem, nullptr, vb, nullptr);
  }
}

// bidx[r * 33 + k] = index into vals_full of K_free[r][r - k] (k = 0..32), -1 off the pattern (the slots k_band_gather
// fills in the dense band Ab of the shared-matrix factor)
__global__ void k_bps_bidx(const MeshDev M, int npad, int* __restrict__ bidx) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= npad) return;
  int* row = bidx + static_cast<size_t>(r) * (BW + 1);
  for (int k = 0; k <= BW; ++k) row[k] = -1;
  if (r >= M.n_free) return;
  for (int k = M.rowptr_f[r]; k < M.rowptr_f[r + 1]; ++k) {
    const int c = M.col_f[k];
    if (c <= r) row[r - c] = M.src_f[k];
  }
}

// K_free(kappa_b) = L_b L_b^T, one CTA per sample.  The dense block Cholesky, X = S L^{-T} and the rank-32 update compute
// every entry with the operations, in the order, of k_band_factor_blk (dfe_batch.cu: see the algorithm there); only the
// loops over the entries of a block are spread over FT instead of 256 threads, which changes no entry's arithmetic.
// Several CTAs share an SM: the one-warp pivot chains of different samples overlap.
//   out = invd[npad] | Lr[npad * 32] of sample b (the layout of dfe_band_factor)
__global__ void __launch_bounds__(FT, 4) k_bps_factor(int n, int npad, const double* __restrict__ vals, long long vstride,
                                                      const int* __restrict__ bidx, double* __restrict__ out,
                                                      int* __restrict__ status) {
  __shared__ double Ls[32][33];
  __shared__ double Xs[32][33];
  __shared__ double Ns[2][32][33];
  __shared__ double Ss[32][33];
  __shared__ double sinv[32];
  __shared__ int sbad;
  const long long smp = blockIdx.x;
  const double* vb = vals + smp * vstride;
  double* invd = out + smp * (static_cast<long long>(npad) * (BW + 1));
  double* Lr = invd + npad;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = npad >> 5;
  // Ab[r * 33 + k] of the shared-matrix kernel, read through the pattern (rows r < n only)
  auto ab = [&](int r, int k) {
    const int i = bidx[static_cast<size_t>(r) * (BW + 1) + k];
    return i >= 0 ? vb[i] : 0.0;
  };
  auto load_diag = [&](int k) {
    for (int q = tid; q < 1024; q += FT) {
      const int a = q >> 5, b = q & 31;
      const int r = 32 * k + a;
      double v = 0.0;
      if (b <= a) v = r < n ? ab(r, a - b) : (a == b ? 1.0 : 0.0);
      Ns[k & 1][a][b] = v;
    }
  };
  if (tid == 0) sbad = 0;
  // entries of block row 0 that would couple to a block row -1 (dfe_band_factor leaves them at its memset's zero)
  for (int q = tid; q < 1024; q += FT) {
    const int aa = q >> 5, b = q & 31;
    if (b >= aa) Lr[static_cast<size_t>(aa) * BW + (32 + aa - b) - 1] = 0.0;
  }
  load_diag(0);
  for (int k = 0; k < nb; ++k) {
    const int cur = k & 1;
    __syncthreads();
    if (warp == 0) {
      double a[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) a[c] = Ns[cur][lane][c];
      const int r = 32 * k + lane;
      const double d0 = r < n ? ab(r, 0) : 1.0;
      bool bad = false;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const double pj = __shfl_sync(FULL, a[j], j);
        const double dj = __shfl_sync(FULL, d0, j);
        const bool ok = pj > 1e-12 * dj;
        bad = bad || !ok;
        const double inv = ok ? rsqrt(pj) : 1.0;
        const double lij = a[j] * inv;
        a[j] = lij;
        if (lane == j) sinv[j] = inv;
#pragma unroll
        for (int m = j + 1; m < 32; ++m) {
          const double lmj = __shfl_sync(FULL, lij, m);
          a[m] = fma(-lij, lane >= m ? lmj : 0.0, a[m]);
        }
      }
      if (bad && lane == 0) sbad = 1;
#pragma unroll
      for (int c = 0; c < 32; ++c) Ls[lane][c] = c <= lane ? a[c] : 0.0;
    } else {
      for (int q = tid - 32; q < 1024; q += FT - 32) {
        const int aa = q >> 5, b = q & 31;
        const int r = 32 * (k + 1) + aa;
        Ss[aa][b] = (k + 1 < nb && b >= aa && r < n) ? ab(r, 32 + aa - b) : 0.0;
        double v = 0.0;
        if (k + 1 < nb && b <= aa) v = r < n ? ab(r, aa - b) : (aa == b ? 1.0 : 0.0);
        Ns[cur ^ 1][aa][b] = v;
      }
    }
    __syncthreads();
    if (warp == 0) {
      double x[32];
#pragma unroll
      for (int b = 0; b < 32; ++b) x[b] = Ss[lane][b];
#pragma unroll
      for (int b = 0; b < 32; ++b) {
        double acc = x[b];
#pragma unroll
        for (int c = 0; c < b; ++c) acc = fma(-x[c], Ls[b][c], acc);
        x[b] = acc * sinv[b];
      }
#pragma unroll
      for (int b = 0; b < 32; ++b) Xs[lane][b] = x[b];
    } else {
      for (int q = tid - 32; q < 1024; q += FT - 32) {
        const int i = q >> 5, j = q & 31;
        const size_t gi = static_cast<size_t>(32 * k + i);
        if (i == j) invd[gi] = sinv[i];
        if (i > j) Lr[gi * BW + (i - j) - 1] = Ls[i][j];
      }
    }
    __syncthreads();
    if (k + 1 < nb) {
      for (int q = tid; q < 1024; q += FT) {
        const int aa = q >> 5, b = q & 31;
        if (b <= aa) {
          double acc = Ns[cur ^ 1][aa][b];
#pragma unroll 8
          for (int c = 0; c < 32; ++c) acc = fma(-Xs[aa][c], Xs[b][c], acc);
          Ns[cur ^ 1][aa][b] = acc;
        }
        if (b >= aa) Lr[static_cast<size_t>(32 * (k + 1) + aa) * BW + (32 + aa - b) - 1] = Xs[aa][b];
      }
    }
  }
  __syncthreads();
  if (tid == 0) status[smp] = sbad ? 5 : 0;
}

// L_b y = b, L_b^T x = y for one right-hand side per factor: one warp per sample, both sweeps of bps_sweeps
// (dfe_band_ps_solve.cuh).  GIN: the right-hand side is gathered from gsrc (B, ldg) through the free-node table (the
// adjoint's gbar); SOUT: x is scattered into u (B, ldu) with the Dirichlet values (the forward solution); otherwise both are
// in X (B, npad), free numbering.
template <bool GIN, bool SOUT>
__global__ void __launch_bounds__(32 * SW_) k_bps_solve(const MeshDev M, long long B, int npad,
                                                        const double* __restrict__ fac, double* __restrict__ X,
                                                        const double* __restrict__ gsrc, long long ldg,
                                                        double* __restrict__ uout, long long ldu) {
  const int lane = threadIdx.x & 31;
  const long long b = blockIdx.x * static_cast<long long>(SW_) + (threadIdx.x >> 5);
  if (b >= B) return;
  const double* invd = fac + b * (static_cast<long long>(npad) * (BW + 1));
  double* x = X + b * npad;
  const int n = M.n_free;
  bps_sweeps(
      invd, invd + npad, x, npad >> 5, lane,
      [&](int i) { return GIN ? (i < n ? gsrc[b * ldg + M.free_nodes[i]] : 0.0) : x[i]; },
      [&](int i, double xv) {
        if (SOUT) {
          if (i < n) uout[b * ldu + M.free_nodes[i]] = xv;
        } else {
          x[i] = xv;
        }
      });
  if (SOUT)
    for (int d = lane; d < M.n_dir; d += 32) uout[b * ldu + M.dir_idx[d]] = M.dir_val[d];   // solver.py:177-179
}

inline unsigned nblk(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

bool ps_fits(const dfe_mesh* m) { return m && m->info.device >= 0 && m->dev.dim == 2 && dfe_band_supported(m); }

size_t ps_tables(const dfe_mesh* m) { return 12 * static_cast<size_t>(m->dev.n_el); }   // geom | geom2, doubles
size_t ps_sample(const dfe_mesh* m) { return static_cast<size_t>(dfe_band_npad(m)) * (BW + 1); }

int ps_enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (!ps_fits(m)) {
    dfe::set_error("%s: needs a 2-D P1 mesh whose K_free has half bandwidth <= %d (dfe_band_supported)", who, BW);
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}

}  // namespace

void dfe::band_ps_assemble(const dfe_mesh* m, long long B, const double* kappa, int per_elem, double* vals,
                           cudaStream_t st) {
  const dim3 ag(nblk(m->dev.n_nodes, 128), static_cast<unsigned>(B < 65535 ? B : 65535));
  k_bps_assemble<<<ag, 128, 0, st>>>(m->dev, B, kappa, per_elem, vals);
}

void dfe::band_ps_factor(const dfe_mesh* m, long long B, const double* vals, long long vstride, int* bidx, double* fac,
                         int* status, cudaStream_t st) {
  const int np = static_cast<int>(dfe_band_npad(m));
  k_bps_bidx<<<nblk(np, 128), 128, 0, st>>>(m->dev, np, bidx);
  k_bps_factor<<<static_cast<unsigned>(B), FT, 0, st>>>(m->dev.n_free, np, vals, vstride, bidx, fac, status);
}

extern "C" int dfe_band_ps_supported(const dfe_mesh* m) { return ps_fits(m) ? 1 : 0; }

extern "C" size_t dfe_band_ps_factor_bytes(const dfe_mesh* m, int64_t B) {
  if (!ps_fits(m) || B < 1) return 0;
  return (ps_tables(m) + static_cast<size_t>(B) * ps_sample(m)) * sizeof(double);
}

extern "C" size_t dfe_band_ps_workspace_bytes(const dfe_mesh* m, int64_t B) {
  if (!ps_fits(m) || B < 1) return 0;
  const size_t np = static_cast<size_t>(dfe_band_npad(m));
  // vals_full (B, nnz_full) | X (B, npad) | bidx (npad, 33) int32
  return static_cast<size_t>(B) * (static_cast<size_t>(m->dev.nnz_full) + np) * sizeof(double) + np * (BW + 1) * sizeof(int);
}

extern "C" int dfe_band_ps_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* kappa,
                               int kappa_mode, void* factors, double* u, int64_t ldu, int32_t* status, void* ws,
                               size_t ws_bytes, void* stream) {
  int prev;
  int rc = ps_enter(m, "dfe_band_ps_fwd", &prev);
  if (rc) return rc;
  if (!f || !kappa || !factors || !u || !status || !ws || B < 1 || ldf < m->dev.n_nodes || ldu < m->dev.n_nodes) {
    dfe::set_error("dfe_band_ps_fwd: null / invalid argument (row strides must be >= n_nodes)");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_PER_SAMPLE && kappa_mode != DFE_KAPPA_PER_SAMPLE_ELEMENT) {
    dfe::set_error("dfe_band_ps_fwd: kappa_mode must be PER_SAMPLE or PER_SAMPLE_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_band_ps_workspace_bytes(m, B)) {
    dfe::set_error("dfe_band_ps_fwd: workspace %zu bytes < required %zu", ws_bytes, dfe_band_ps_workspace_bytes(m, B));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int np = static_cast<int>(dfe_band_npad(m));
    double* geom = static_cast<double*>(factors);
    double* geom2 = geom + 8 * static_cast<size_t>(m->dev.n_el);
    double* fac = geom + ps_tables(m);
    double* vals = static_cast<double*>(ws);
    double* X = vals + static_cast<size_t>(B) * m->dev.nnz_full;
    int* bidx = reinterpret_cast<int*>(X + static_cast<size_t>(B) * np);
    dfe::band_tables(m, geom, geom2, st);
    dfe::band_ps_assemble(m, B, kappa, kappa_mode == DFE_KAPPA_PER_SAMPLE_ELEMENT, vals, st);
    dfe::band_ps_factor(m, B, vals, m->dev.nnz_full, bidx, fac, status, st);
    dfe::band_rhs(m, B, f, ldf, vals, m->dev.nnz_full, geom, X, st);
    k_bps_solve<false, true><<<nblk(B, SW_), 32 * SW_, 0, st>>>(m->dev, B, np, fac, X, nullptr, 0, u, ldu);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      dfe::set_error("dfe_band_ps_fwd: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_band_ps_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                               const void* factors, int kappa_mode, double* gf, int64_t ldgf, double* gkappa, void* ws,
                               size_t ws_bytes, void* stream) {
  int prev;
  int rc = ps_enter(m, "dfe_band_ps_bwd", &prev);
  if (rc) return rc;
  if (!gbar || !u || !factors || !gkappa || !ws || B < 1 || ldg < m->dev.n_nodes || ldu < m->dev.n_nodes ||
      (gf && ldgf < m->dev.n_nodes)) {
    dfe::set_error("dfe_band_ps_bwd: null / invalid argument (row strides must be >= n_nodes)");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_PER_SAMPLE && kappa_mode != DFE_KAPPA_PER_SAMPLE_ELEMENT) {
    dfe::set_error("dfe_band_ps_bwd: kappa_mode must be PER_SAMPLE or PER_SAMPLE_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_band_ps_workspace_bytes(m, B)) {
    dfe::set_error("dfe_band_ps_bwd: workspace %zu bytes < required %zu", ws_bytes, dfe_band_ps_workspace_bytes(m, B));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int np = static_cast<int>(dfe_band_npad(m));
    const double* geom = static_cast<const double*>(factors);
    const double* geom2 = geom + 8 * static_cast<size_t>(m->dev.n_el);
    const double* fac = geom + ps_tables(m);
    double* X = static_cast<double*>(ws);
    k_bps_solve<true, false><<<nblk(B, SW_), 32 * SW_, 0, st>>>(m->dev, B, np, fac, X, gbar, ldg, nullptr, 0);
    rc = dfe::band_grad(m, B, X, u, ldu, geom, geom2, kappa_mode == DFE_KAPPA_PER_SAMPLE_ELEMENT, gkappa, gf, ldgf, st);
    cudaError_t e = cudaGetLastError();
    if (rc == DFE_OK && e != cudaSuccess) {
      dfe::set_error("dfe_band_ps_bwd: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}
