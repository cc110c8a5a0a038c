// Batched solve / adjoint of MANY small systems that share one matrix (kappa shared by the batch: a scalar or a
// per-element field) on a general mesh — BASELINE config 5b: 65 536 forcing samples on rectangle(32, 32).
//
// Replaces, for every sample b, solver.py:143-145 (load), :165-169 (lifting), :174 (torch.linalg.solve),
// :177-181 (scatter) and the autograd backward of those (SURVEY §8a rows A5-A8).  The per-sample route
// (dfe_assemble + dfe_eliminate + dfe_pcg, one cooperative whole-GPU kernel and a stream synchronisation per
// system) is latency-bound at this size; here ONE CTA owns a sample: the SELL-32 copy of K_free (values and
// columns) and the search direction p live in shared memory, x / r / q / 1/diag in registers (a thread owns the
// same rows for the whole solve), the dot products are fixed-order block reductions (bit-reproducible, no float
// atomics), and a CTA loops over samples b = blockIdx, blockIdx + grid, ...  The matrix is loaded once per CTA.
//
//   forward   F_b (node-centred gather in ascending element order, the arithmetic of k_assemble) -> lifting in
//             dict order (the arithmetic of k_eliminate) -> Jacobi-PCG to the recursive tolerance -> scatter
//   adjoint   lambda_b = K_free^{-1} gbar_b[free] -> dL/dkappa (per element, or summed per sample) and dL/df_b
#include <cstdlib>

#include "dfe_internal.h"

namespace {

using dfe::MeshDev;
#include "dfe_1d_common.cuh"        // mbarrier / 1-D TMA bulk copy wrappers (used by the tensor-core band solve)
#include "dfe_band_mma.cuh"         // block-row step of the tensor-core band solve and its fragment layout
#include "dfe_exact.cuh"            // div3: correctly rounded x / 3.0 without the division instruction

constexpr double AREA_EPS = 1e-15;  // solver.py:120
constexpr int BT = 256;             // threads per CTA (few warps: the per-warp scalar work of CG — reductions, alpha,
                                    // beta — is replicated in every warp, and this kernel is bound by instruction issue)
constexpr int BNW = BT / 32;
constexpr int RPT_MAX = 8;          // SELL slices per warp  =>  n_free <= 32 * BNW * RPT_MAX = 2048
constexpr int WMAX = 8;             // SELL slice widths up to WMAX are unrolled (wider slices take the generic loop)

struct BArgs {
  MeshDev M;
  long long B;
  const double* in;        // forward: f (B, n_nodes); adjoint: gbar (B, n_nodes)
  long long ldin;
  const double* u;         // adjoint: forward solution (B, n_nodes)
  long long ldu;
  const double* vals_full; // forward: assembled K on the full pattern (lifting terms)
  const double* sell_vals;
  const double* dinv;
  double* out;             // forward: u ; adjoint: dL/df (may be null)
  long long ldout;
  double* gk;              // adjoint: (B) [scalar kappa] or (B, n_el) [per-element kappa]
  int gk_per_elem;
  double tol;
  int maxit;
  int* iters;              // (B)
  double* relres;          // (B)
  int* status;             // (B): 0 ok, 4 not converged, 5 breakdown
};

struct Elem2D {
  double area, b[3], c[3];
};
// solver.py:114-134 in the reference's operation order (same as dfe_general.cu)
__device__ __forceinline__ Elem2D elem2d(const MeshDev& M, int e, int n[3]) {
  n[0] = M.elems[3 * e + 0];
  n[1] = M.elems[3 * e + 1];
  n[2] = M.elems[3 * e + 2];
  const double xi = M.nodes[2 * n[0]], yi = M.nodes[2 * n[0] + 1];
  const double xj = M.nodes[2 * n[1]], yj = M.nodes[2 * n[1] + 1];
  const double xk = M.nodes[2 * n[2]], yk = M.nodes[2 * n[2] + 1];
  Elem2D E;
  const double cr = __dsub_rn(__dmul_rn(__dsub_rn(xj, xi), __dsub_rn(yk, yi)), __dmul_rn(__dsub_rn(xk, xi), __dsub_rn(yj, yi)));
  E.area = __dmul_rn(0.5, fabs(cr));
  E.b[0] = __dsub_rn(yj, yk);
  E.b[1] = __dsub_rn(yk, yi);
  E.b[2] = __dsub_rn(yi, yj);
  E.c[0] = __dsub_rn(xk, xj);
  E.c[1] = __dsub_rn(xi, xk);
  E.c[2] = __dsub_rn(xj, xi);
  return E;
}

// F_p of one node (solver.py:95-96 / :143-145), accumulated over the adjacent elements in ascending element order
__device__ __forceinline__ double load_at(const MeshDev& M, const double* f, int p) {
  double Fp = 0.0;
  for (int a = M.adj_ptr[p]; a < M.adj_ptr[p + 1]; ++a) {
    const int e = M.adj_elem[a];
    if (M.dim == 1) {
      const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
      const double h = __dsub_rn(M.nodes[j], M.nodes[i]);
      Fp = __dadd_rn(Fp, __dmul_rn(__ddiv_rn(h, 2.0), f[p]));
    } else {
      int n[3];
      const Elem2D E = elem2d(M, e, n);
      if (E.area < AREA_EPS) continue;
      const double fc = __ddiv_rn(__dadd_rn(__dadd_rn(f[n[0]], f[n[1]]), f[n[2]]), 3.0);
      Fp = __dadd_rn(Fp, __dmul_rn(__ddiv_rn(E.area, 3.0), fc));
    }
  }
  return Fp;
}

// fixed-order block sums of up to two values; every thread returns the same bits
__device__ __forceinline__ void block_sum2(double& a, double& b, double* sh, int lane, int warp) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, d);
    b += __shfl_xor_sync(0xffffffffu, b, d);
  }
  if (lane == 0) { sh[2 * warp] = a; sh[2 * warp + 1] = b; }
  __syncthreads();
  // every warp folds the BNW partials with the same butterfly (lane l holds partial l mod BNW): same bits everywhere
  double x = sh[2 * (lane & (BNW - 1))], y = sh[2 * (lane & (BNW - 1)) + 1];
#pragma unroll
  for (int d = BNW / 2; d > 0; d >>= 1) {
    x += __shfl_xor_sync(0xffffffffu, x, d);
    y += __shfl_xor_sync(0xffffffffu, y, d);
  }
  a = x;
  b = y;
}

// block max of non-negative values (a max is exact in any order); every thread returns the same bits
__device__ __forceinline__ double block_max(double a, double* sh, int lane, int warp) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) a = fmax(a, __shfl_xor_sync(0xffffffffu, a, d));
  if (lane == 0) sh[warp] = a;
  __syncthreads();
  double x = sh[lane & (BNW - 1)];
#pragma unroll
  for (int d = BNW / 2; d > 0; d >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, d));
  return x;
}

template <bool BWD, int RPT>
__global__ void __launch_bounds__(BT, (RPT <= 4 ? 2 : 1)) k_batch(const BArgs A) {
  extern __shared__ __align__(16) unsigned char smem[];
  const MeshDev& M = A.M;
  const int n = M.n_free, nsl = M.n_slices;
  double* sval = reinterpret_cast<double*>(smem);                 // [sell_nnz]
  double* sp = sval + M.sell_nnz;                                  // [32 * n_slices] search direction
  double* sred = sp + 32 * nsl;                                    // [3][2 * BNW]
  double* slam = sred + 6 * BNW;                                   // adjoint: [n_nodes] lambda on all nodes
  int* scol = reinterpret_cast<int*>(slam + (BWD ? M.n_nodes : 0));   // [sell_nnz]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  for (int k = tid; k < M.sell_nnz; k += BT) {
    sval[k] = A.sell_vals[k];
    scol[k] = M.sell_col[k];
  }
  // rows owned by this thread: slice warp + BNW * j, lane
  int row[RPT], beg[RPT], wd[RPT];
  double dinv[RPT];
#pragma unroll
  for (int j = 0; j < RPT; ++j) {
    const int s = warp + BNW * j;
    const bool on = s < nsl && 32 * s + lane < n;
    row[j] = on ? 32 * s + lane : -1;
    beg[j] = s < nsl ? M.slice_ptr[s] : 0;
    wd[j] = s < nsl ? (M.slice_ptr[s + 1] - M.slice_ptr[s]) >> 5 : 0;
    dinv[j] = on ? A.dinv[row[j]] : 0.0;
  }
  __syncthreads();

  for (long long b = blockIdx.x; b < A.B; b += gridDim.x) {
    const double* in = A.in + b * A.ldin;
    // ---- right-hand side
    double x[RPT], r[RPT], z[RPT], p[RPT], q[RPT];
    double amax = 0.0;
#pragma unroll
    for (int j = 0; j < RPT; ++j) {
      x[j] = r[j] = z[j] = p[j] = q[j] = 0.0;
      if (row[j] >= 0) {
        const int node = M.free_nodes[row[j]];
        double Fr;
        if (BWD) {
          Fr = in[node];                                           // gbar restricted to the free rows (SURVEY A7)
        } else {
          Fr = load_at(M, in, node);
          for (int t = M.lift_ptr[row[j]]; t < M.lift_ptr[row[j] + 1]; ++t)
            Fr = __dsub_rn(Fr, __dmul_rn(A.vals_full[M.lift_src[t]], M.lift_g[t]));   // solver.py:169
        }
        r[j] = Fr;
        amax = fmax(amax, fabs(Fr));
      }
    }
    // Solve for 2^sc * Fr with max |2^sc Fr| in [1, 2): the squares in ||Fr||^2, tol^2 ||Fr||^2 and p.q then neither
    // underflow (|Fr| < ~2e-162 would give bb == 0, i.e. "converged" at x = 0; below ~1e-154 tol^2 bb underflows and the
    // loop stops far above tol) nor overflow.  Scaling by a power of two is exact, so where no intermediate leaves the
    // normal range the iterates are those of the unscaled solve, scaled.
    amax = block_max(amax, sred + 2 * BNW, lane, warp);
    int sc = 0;
    if (amax > 0.0 && isfinite(amax)) {    // (0: nothing to solve; inf / NaN: reported as a breakdown below)
      frexp(amax, &sc);
      sc = 1 - sc;
    }
    double bb = 0.0, rz = 0.0;
#pragma unroll
    for (int j = 0; j < RPT; ++j) {
      if (row[j] >= 0) {
        const double Fr = ldexp(r[j], sc);
        r[j] = Fr;
        z[j] = dinv[j] * Fr;
        p[j] = z[j];
        bb = fma(Fr, Fr, bb);
        rz = fma(Fr, z[j], rz);
      }
      if (warp + BNW * j < nsl) sp[32 * (warp + BNW * j) + lane] = p[j];
    }
    block_sum2(bb, rz, sred, lane, warp);   // (its barrier also publishes sp)
    const double tol2bb = (A.tol * A.tol) * bb;
    int status = 0, it = 0;
    double rr_last = 0.0;
    if (!(bb > 0.0)) {
      if (bb != 0.0) status = 5;            // non-finite right-hand side
    } else {
      status = 4;
      while (it < A.maxit) {
        // ---- q = K p (SELL-32 from shared memory), p.q
        double pq = 0.0, dummy = 0.0;
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          double sum = 0.0;
          if (wd[j] <= WMAX) {   // all loads of the row first (independent), then the fma chain in column order
            double v[WMAX], g[WMAX];
#pragma unroll
            for (int w = 0; w < WMAX; ++w) {
              const int k = beg[j] + (w << 5) + lane;
              const bool on = w < wd[j];
              v[w] = on ? sval[k] : 0.0;
              g[w] = on ? sp[scol[k]] : 0.0;
            }
#pragma unroll
            for (int w = 0; w < WMAX; ++w)
              if (w < wd[j]) sum = fma(v[w], g[w], sum);
          } else {
            for (int w = 0; w < wd[j]; ++w) {
              const int k = beg[j] + (w << 5) + lane;
              sum = fma(sval[k], sp[scol[k]], sum);
            }
          }
          q[j] = sum;
          if (row[j] >= 0) pq = fma(p[j], sum, pq);
        }
        block_sum2(pq, dummy, sred + 2 * BNW, lane, warp);
        if (!(pq > 0.0) || !isfinite(pq)) { status = 5; break; }
        const double alpha = rz / pq;
        // ---- x, r, z, r.z, r.r
        double rzn = 0.0, rr = 0.0;
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          if (row[j] >= 0) {
            x[j] = fma(alpha, p[j], x[j]);
            r[j] = fma(-alpha, q[j], r[j]);
            z[j] = dinv[j] * r[j];
            rzn = fma(r[j], z[j], rzn);
            rr = fma(r[j], r[j], rr);
          }
        }
        block_sum2(rzn, rr, sred + 4 * BNW, lane, warp);
        ++it;
        rr_last = rr;
        if (!isfinite(rr)) { status = 5; break; }
        if (rr <= tol2bb) { status = 0; break; }      // ||r|| <= tol ||b||, squared: no sqrt / division in the loop
        const double beta = rzn / rz;
        rz = rzn;
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          if (row[j] >= 0) {
            p[j] = fma(beta, p[j], z[j]);
            sp[row[j]] = p[j];
          }
        }
        __syncthreads();
      }
    }
    if (tid == 0) {
      A.iters[b] = it;
      A.relres[b] = bb > 0.0 ? sqrt(rr_last / bb) : 0.0;
      A.status[b] = status;
    }
    if (!BWD) {
      // ---- u = 0; u[d] = g; u[free] = 2^-sc x   (solver.py:177-181)
      double* u = A.out + b * A.ldout;
#pragma unroll
      for (int j = 0; j < RPT; ++j)
        if (row[j] >= 0) u[M.free_nodes[row[j]]] = ldexp(x[j], -sc);
      for (int i = tid; i < M.n_dir; i += BT) u[M.dir_idx[i]] = M.dir_val[i];
    } else {
      // ---- lambda on all nodes (0 on Dirichlet nodes), then the closed-form backward of the assembly (SURVEY A8)
      __syncthreads();   // every thread left the solve loop: slam / sred are free
      for (int i = tid; i < M.n_nodes; i += BT) slam[i] = 0.0;
      __syncthreads();
#pragma unroll
      for (int j = 0; j < RPT; ++j)
        if (row[j] >= 0) slam[M.free_nodes[row[j]]] = ldexp(x[j], -sc);
      __syncthreads();
      const double* u = A.u + b * A.ldu;
      double gsum = 0.0, dummy = 0.0;
      for (int e = tid; e < M.n_el; e += BT) {
        double g = 0.0;
        if (M.dim == 1) {
          const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
          const double h = M.nodes[j] - M.nodes[i];
          g = -(slam[j] - slam[i]) * (u[j] - u[i]) / h;
        } else {
          int nd[3];
          const Elem2D E = elem2d(M, e, nd);
          if (!(E.area < AREA_EPS)) {
            double bl = 0, bu = 0, cl = 0, cu = 0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              const double l = slam[nd[c]], uu = u[nd[c]];
              bl = fma(E.b[c], l, bl);
              bu = fma(E.b[c], uu, bu);
              cl = fma(E.c[c], l, cl);
              cu = fma(E.c[c], uu, cu);
            }
            g = -(bl * bu + cl * cu) / (4.0 * E.area);
          }
        }
        if (A.gk_per_elem) A.gk[b * M.n_el + e] = g;
        else gsum += g;
      }
      if (!A.gk_per_elem) {
        block_sum2(gsum, dummy, sred, lane, warp);
        if (tid == 0) A.gk[b] = gsum;
      }
      if (A.out) {
        double* gf = A.out + b * A.ldout;
        for (int pn = tid; pn < M.n_nodes; pn += BT) {
          double g = 0.0;
          for (int a = M.adj_ptr[pn]; a < M.adj_ptr[pn + 1]; ++a) {
            const int e = M.adj_elem[a];
            if (M.dim == 1) {
              const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
              g = fma((M.nodes[j] - M.nodes[i]) * 0.5, slam[pn], g);
            } else {
              int nd[3];
              const Elem2D E = elem2d(M, e, nd);
              if (E.area < AREA_EPS) continue;
              g = fma(E.area / 9.0, (slam[nd[0]] + slam[nd[1]]) + slam[nd[2]], g);
            }
          }
          gf[pn] = g;
        }
      }
    }
    __syncthreads();   // sp / sred / slam are reused by the next sample
  }
}

// =====================================================================================================================
// Banded direct solver for the same job when the half bandwidth of K_free is <= 32 (rectangle(nx, ny) with nx <= 32
// in the reference's node numbering): K_free = L L^T once per call (the batch shares the matrix), then two banded
// triangular solves per sample (a block TRSM on the FP64 tensor cores, k_band_solve_mma).  That is ~13x fewer flops
// than ~120 Jacobi-PCG iterations at 961 unknowns and has no reductions.  Replaces solver.py:174 (LU with partial
// pivoting on the dense K_free) more literally than PCG does.
constexpr int BW = 32;   // half bandwidth supported

// Lower band of K_free, Ab[r * 33 + k] = K_free[r][r - k] (k = 0..32), scattered from the assembled matrix in parallel.
// Rows n_free and beyond are zero.
__global__ void k_band_gather(const MeshDev M, const double* __restrict__ vals_full, double* __restrict__ Ab) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= M.n_free) return;
  for (int k = M.rowptr_f[r]; k < M.rowptr_f[r + 1]; ++k) {
    const int c = M.col_f[k];
    if (c <= r) Ab[static_cast<size_t>(r) * (BW + 1) + (r - c)] = vals_full[M.src_f[k]];
  }
}

// K_free = L L^T in ONE CTA, blocked.  (Round 1 factored row by row: ~1500 cycles for each of the n dependent pivot steps
// — two CTA barriers, a shared-memory round trip and a double-precision rsqrt per step: 0.72 ms at 961 unknowns, 18 % of a
// config-5b step and, replicated on every rank, the part that does not scale over GPUs.)  With 32 x 32 blocks the band is
// block tridiagonal:
//     L_kk L_kk^T = A_kk - L_{k,k-1} L_{k,k-1}^T,      L_{k+1,k} = A_{k+1,k} L_kk^{-T}.
// The dense Cholesky of a diagonal block runs in ONE warp out of registers (lane i holds row i; pivots and multipliers
// move by shuffles with compile-time register indices, no barrier and no shared-memory latency in the pivot chain), the
// triangular solve for L_{k+1,k} in the same warp (lane a holds row a; L_kk is read from shared memory as broadcasts),
// and the rank-32 update of the next diagonal block by the whole CTA — three CTA barriers per BLOCK.
//   invd[i] = 1 / L_ii,  Lr[i*32 + d-1] = L[i][i-d]   (d = 1..32; rows >= n: identity)
__global__ void __launch_bounds__(256) k_band_factor_blk(int n, int npad, const double* __restrict__ Ab,
                                                         double* __restrict__ invd, double* __restrict__ Lr,
                                                         int* __restrict__ status) {
  __shared__ double Ls[32][33];   // L_kk (lower triangle, diagonal included)
  __shared__ double Xs[32][33];   // L_{k+1,k}: Xs[a][b] = L[32(k+1)+a][32k+b] (zero for b < a)
  __shared__ double Ns[2][32][33];   // diagonal blocks k / k+1 (ping-pong): raw, then minus the rank-32 update (lower triangle)
  __shared__ double Ss[32][33];   // A_{k+1,k}: Ss[a][b] = A[32(k+1)+a][32k+b] (zero for b < a)
  __shared__ double sinv[32];
  __shared__ int sbad;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = npad >> 5;
  constexpr unsigned FULL = 0xffffffffu;
  auto load_diag = [&](int k) {   // Ns <- A_kk (lower; identity on the padding rows), by every thread of the CTA
    for (int q = tid; q < 1024; q += 256) {
      const int a = q >> 5, b = q & 31;
      const int r = 32 * k + a;
      double v = 0.0;
      if (b <= a) v = r < n ? Ab[static_cast<size_t>(r) * (BW + 1) + (a - b)] : (a == b ? 1.0 : 0.0);
      Ns[k & 1][a][b] = v;
    }
  };
  if (tid == 0) sbad = 0;
  load_diag(0);
  for (int k = 0; k < nb; ++k) {
    const int cur = k & 1;
    __syncthreads();   // [B1] Ns[cur] = diagonal block k, updated
    if (warp == 0) {
      // ---- dense Cholesky of the block, row `lane` in registers
      double a[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) a[c] = Ns[cur][lane][c];
      const int r = 32 * k + lane;
      const double d0 = r < n ? Ab[static_cast<size_t>(r) * (BW + 1)] : 1.0;   // diagonal entry before elimination
      bool bad = false;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const double pj = __shfl_sync(FULL, a[j], j);
        const double dj = __shfl_sync(FULL, d0, j);
        // SPD check: a pivot that lost 12 digits against its diagonal entry means K_free is (numerically) singular
        const bool ok = pj > 1e-12 * dj;
        bad = bad || !ok;
        const double inv = ok ? rsqrt(pj) : 1.0;
        const double lij = a[j] * inv;        // L[i][j] for i >= j (lane j: L_jj = p_j / sqrt(p_j))
        a[j] = lij;
        if (lane == j) sinv[j] = inv;
#pragma unroll
        for (int m = j + 1; m < 32; ++m) {
          const double lmj = __shfl_sync(FULL, lij, m);
          a[m] = fma(-lij, lane >= m ? lmj : 0.0, a[m]);   // (a select, not a predicated store: keeps a[] in registers)
        }
      }
      if (bad && lane == 0) sbad = 1;
#pragma unroll
      for (int c = 0; c < 32; ++c) Ls[lane][c] = c <= lane ? a[c] : 0.0;
    } else {
      // ---- meanwhile: the blocks of the next block row
      for (int q = tid - 32; q < 1024; q += 224) {
        const int aa = q >> 5, b = q & 31;
        const int r = 32 * (k + 1) + aa;
        Ss[aa][b] = (k + 1 < nb && b >= aa && r < n) ? Ab[static_cast<size_t>(r) * (BW + 1) + (32 + aa - b)] : 0.0;
        double v = 0.0;
        if (k + 1 < nb && b <= aa) v = r < n ? Ab[static_cast<size_t>(r) * (BW + 1) + (aa - b)] : (aa == b ? 1.0 : 0.0);
        Ns[cur ^ 1][aa][b] = v;
      }
    }
    __syncthreads();   // [B2] Ls, sinv, Ss, raw Ns[cur ^ 1] ready
    if (warp == 0) {
      // ---- X = S L^{-T}: row `lane` of S in registers, forward substitution along the row
      double x[32];
#pragma unroll
      for (int b = 0; b < 32; ++b) x[b] = Ss[lane][b];
#pragma unroll
      for (int b = 0; b < 32; ++b) {
        double acc = x[b];   // (four partial accumulators were measured: 383 -> 410 us, the chain is not the limiter)
#pragma unroll
        for (int c = 0; c < b; ++c) acc = fma(-x[c], Ls[b][c], acc);
        x[b] = acc * sinv[b];
      }
#pragma unroll
      for (int b = 0; b < 32; ++b) Xs[lane][b] = x[b];
    } else {
      // ---- meanwhile: the factor entries inside the diagonal block
      for (int q = tid - 32; q < 1024; q += 224) {
        const int i = q >> 5, j = q & 31;
        const size_t gi = static_cast<size_t>(32 * k + i);
        if (i == j) invd[gi] = sinv[i];
        if (i > j) Lr[gi * BW + (i - j) - 1] = Ls[i][j];
      }
    }
    __syncthreads();   // [B3] Xs ready
    if (k + 1 < nb) {
      for (int q = tid; q < 1024; q += 256) {
        const int aa = q >> 5, b = q & 31;
        if (b <= aa) {   // A_{k+1,k+1} -= L_{k+1,k} L_{k+1,k}^T (lower triangle)
          double acc = Ns[cur ^ 1][aa][b];
#pragma unroll 8
          for (int c = 0; c < 32; ++c) acc = fma(-Xs[aa][c], Xs[b][c], acc);
          Ns[cur ^ 1][aa][b] = acc;
        }
        if (b >= aa)   // factor entries that cross the block boundary: row 32(k+1)+aa, column 32k+b
          Lr[static_cast<size_t>(32 * (k + 1) + aa) * BW + (32 + aa - b) - 1] = Xs[aa][b];
      }
    }
  }
  __syncthreads();
  if (tid == 0) *status = sbad ? 5 : 0;
}

// Per-element constants shared by every sample of the batch (8 doubles per element):
//   [0] area/3 (load weight, solver.py:143-145; -1 marks a skipped / degenerate element)   [1] area/9 (dL/df weight)
//   [2..4] b_p   [5..7] c_p  (2-D);   1-D: [0] h/2 as the reference rounds it  [1] h/2  [2] h
__global__ void k_band_geom(const MeshDev M, double* __restrict__ geom) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= M.n_el) return;
  const size_t ne = static_cast<size_t>(M.n_el);   // structure of arrays: component k of element e at geom[k * n_el + e]
  double g[8];
  if (M.dim == 1) {
    const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
    const double h = __dsub_rn(M.nodes[j], M.nodes[i]);
    g[0] = __ddiv_rn(h, 2.0);
    g[1] = (M.nodes[j] - M.nodes[i]) * 0.5;
    g[2] = M.nodes[j] - M.nodes[i];
    g[3] = g[4] = g[5] = g[6] = g[7] = 0.0;
  } else {
    int nd[3];
    const Elem2D E = elem2d(M, e, nd);
    const bool skip = E.area < AREA_EPS;
    g[0] = skip ? -1.0 : __ddiv_rn(E.area, 3.0);
    g[1] = skip ? -1.0 : E.area / 9.0;
    g[2] = E.b[0]; g[3] = E.b[1]; g[4] = E.b[2];
    g[5] = E.c[0]; g[6] = E.c[1]; g[7] = E.c[2];
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) geom[k * ne + e] = g[k];
}

// right-hand sides of the whole batch, (B, npad) row-major, rows >= n_free zero.
// forward: one CTA per sample — f_b and the per-element terms (area/3) * (f_i+f_j+f_k)/3 (solver.py:143-145) in shared
// memory, then every free row adds the terms of its adjacent elements in ascending element order and applies the
// lifting in dict order (solver.py:165-169): the arithmetic of k_assemble / k_eliminate, bit for bit.  Sample b reads its
// matrix at vals_full + b * vstride (0: one matrix shared by the batch)
__global__ void __launch_bounds__(BT) k_band_rhs_fwd(const MeshDev M, long long B, int npad, const double* __restrict__ f,
                                                     long long ldf, const double* __restrict__ vals_full, long long vstride,
                                                     const double* __restrict__ geom, double* __restrict__ X) {
  extern __shared__ double sg[];
  double* sf = sg;               // [n_nodes]
  double* st = sf + M.n_nodes;   // [n_el]
  const int tid = threadIdx.x;
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    const double* fb = f + b * ldf;
    for (int p = tid; p < M.n_nodes; p += BT) sf[p] = fb[p];
    __syncthreads();
    if (M.dim == 2)
      for (int e = tid; e < M.n_el; e += BT) {
        const double w = geom[e];
        const int n0 = M.elems[3 * e], n1 = M.elems[3 * e + 1], n2 = M.elems[3 * e + 2];
        const double fc = __ddiv_rn(__dadd_rn(__dadd_rn(sf[n0], sf[n1]), sf[n2]), 3.0);
        st[e] = w >= 0.0 ? __dmul_rn(w, fc) : 0.0;   // a skipped element adds nothing
      }
    __syncthreads();
    for (int r = tid; r < npad; r += BT) {
      double v = 0.0;
      if (r < M.n_free) {
        const int node = M.free_nodes[r];
        for (int a = M.adj_ptr[node]; a < M.adj_ptr[node + 1]; ++a) {
          const int e = M.adj_elem[a];
          v = __dadd_rn(v, M.dim == 1 ? __dmul_rn(geom[e], sf[node]) : st[e]);
        }
        for (int t = M.lift_ptr[r]; t < M.lift_ptr[r + 1]; ++t)
          v = __dsub_rn(v, __dmul_rn(vals_full[b * vstride + M.lift_src[t]], M.lift_g[t]));   // solver.py:169
      }
      X[b * npad + r] = v;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Register-resident variant of the gradient kernel (2-D meshes with n_el <= EPT * BT, n_nodes <= NPT * BT — config 5b:
// 2048 / 1089), used when dL/dkappa is wanted PER ELEMENT (a shared per-element kappa field).  k_band_grad above fetches
// connectivity, adjacency and 7 per-element constants from global memory for EVERY sample (launch list: 2.1 ms of a
// 6.4 ms step, 10x its HBM floor).  Here a thread owns the same EPT elements and NPT nodes for the whole batch: their
// indices and constants live in registers, the next sample's rows arrive by cp.async while the current one is processed,
// and a sample costs two CTA barriers.

constexpr int EPT = 8, RPT = 4, NPT = 5;

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// per-factorisation tables: liftp[t] = K[row, d_t] * g_t (the products of the lifting, solver.py:169 — sample
// independent), geom2 = [k01 | k02 | k12 | area/9][n_el] with k_pq = (b_p b_q + c_p c_q) / (4 area), the off-diagonal
// entries of the element matrix at kappa = 1 (zeros for a skipped element)
__global__ void k_band_tables(const MeshDev M, const double* __restrict__ vals_full, int n_lift, double* __restrict__ liftp,
                              double* __restrict__ geom2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_lift) liftp[i] = __dmul_rn(vals_full[M.lift_src[i]], M.lift_g[i]);
  if (i < M.n_el && M.dim == 2) {
    int nd[3];
    const Elem2D E = elem2d(M, i, nd);
    const bool skip = E.area < AREA_EPS;
    const double den = 4.0 * E.area;
    const size_t ne = static_cast<size_t>(M.n_el);
    geom2[i] = skip ? 0.0 : (E.b[0] * E.b[1] + E.c[0] * E.c[1]) / den;
    geom2[ne + i] = skip ? 0.0 : (E.b[0] * E.b[2] + E.c[0] * E.c[2]) / den;
    geom2[2 * ne + i] = skip ? 0.0 : (E.b[1] * E.b[2] + E.c[1] * E.c[2]) / den;
    geom2[3 * ne + i] = skip ? 0.0 : E.area / 9.0;
  }
}

// Where element e keeps its per-sample term in shared memory: even and odd element ids in separate halves, so that the
// rows of consecutive nodes (whose adjacent elements have ids two apart on a rectangle() mesh) hit consecutive banks.
__device__ __forceinline__ int st_slot(int e, int half) { return (e & 1) * half + (e >> 1); }

// The (at most ADJ6) adjacent elements of node `node` in ascending element order as three packed pairs of shared-memory
// slots; missing entries point at the dummy slot `zslot`, which holds +0.0: x + (+0.0) == x bit for bit for every x that
// an accumulation started from +0.0 can reach (it never produces -0.0), so the padded sum has the reference's bits.
constexpr int ADJ6 = 6;
__device__ __forceinline__ void pack_adj(const MeshDev& M, int node, int half, int zslot, unsigned (&pk)[3]) {
  int id[ADJ6];
#pragma unroll
  for (int j = 0; j < ADJ6; ++j) id[j] = zslot;
  if (node >= 0) {
    const int a0 = M.adj_ptr[node], cnt = M.adj_ptr[node + 1] - a0;
    for (int j = 0; j < cnt && j < ADJ6; ++j) id[j] = st_slot(M.adj_elem[a0 + j], half);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) pk[j] = static_cast<unsigned>(id[2 * j]) | (static_cast<unsigned>(id[2 * j + 1]) << 16);
}

// adjoint gradients from lambda = X: dL/dkappa_e = sum_{p<q} k_pq (lam_p - lam_q)(u_p - u_q)  (= -lam^T K_e^0 u for a
// symmetric element matrix with zero row sums), dL/df_q = sum_{e∋q} (area_e / 9) (lam_i + lam_j + lam_k)
__global__ void __launch_bounds__(BT, 2) k_band_grad2(const MeshDev M, long long B, int npad, const double* __restrict__ X,
                                                      const double* __restrict__ ufull, long long ldu,
                                                      const double* __restrict__ geom2, double* __restrict__ gk,
                                                      int gk_per_elem, double* __restrict__ gf, long long ldgf, int nnp) {
  extern __shared__ double sg[];
  double* slam0 = sg;                 // [2][nnp]
  double* su0 = sg + 2 * nnp;         // [2][nnp]
  double* st = sg + 4 * nnp;          // [n_el + 2] (area/9) (lam_i + lam_j + lam_k), then the 0.0 dummy
  const int half = (M.n_el + 1) >> 1, zslot = 2 * half;
  double* sred = st + zslot + 1;      // [2 * BNW]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t ne = static_cast<size_t>(M.n_el);
  if (tid == 0) st[zslot] = 0.0;
  unsigned e01[EPT], e2[EPT];
  double k01[EPT], k02[EPT], k12[EPT], w9[EPT];
#pragma unroll
  for (int k = 0; k < EPT; ++k) {
    const int e = tid + k * BT;
    const bool ex = e < M.n_el;
    e01[k] = ex ? (static_cast<unsigned>(M.elems[3 * e]) | (static_cast<unsigned>(M.elems[3 * e + 1]) << 16)) : 0u;
    e2[k] = ex ? static_cast<unsigned>(M.elems[3 * e + 2]) : 0u;
    k01[k] = ex ? geom2[e] : 0.0;
    k02[k] = ex ? geom2[ne + e] : 0.0;
    k12[k] = ex ? geom2[2 * ne + e] : 0.0;
    w9[k] = ex ? geom2[3 * ne + e] : 0.0;
  }
  unsigned na[NPT][3];         // adjacent element slots of the thread's nodes
  int rk[NPT];
#pragma unroll
  for (int k = 0; k < NPT; ++k) {
    const int p = tid + k * BT;
    rk[k] = -1;
    pack_adj(M, p < M.n_nodes ? p : -1, half, zslot, na[k]);
    if (p < M.n_nodes) {
      rk[k] = M.free_rank[p];
      slam0[p] = 0.0;            // lambda is zero on Dirichlet nodes, in both buffers, for every sample
      slam0[nnp + p] = 0.0;
    }
  }
  long long b = blockIdx.x;
  if (b < B) {
#pragma unroll
    for (int k = 0; k < NPT; ++k) {
      const int p = tid + k * BT;
      if (p < M.n_nodes) {
        su0[p] = ufull[b * ldu + p];
        if (rk[k] >= 0) slam0[p] = X[b * npad + rk[k]];
      }
    }
  }
  __syncthreads();
  int cur = 0;
  for (; b < B; b += gridDim.x) {
    const long long bn = b + gridDim.x;
    const double* lam = slam0 + cur * nnp;
    const double* u = su0 + cur * nnp;
    if (bn < B) {
      double* ln = slam0 + (cur ^ 1) * nnp;
      double* un = su0 + (cur ^ 1) * nnp;
      const double* ug = ufull + bn * ldu;
      const double* xg = X + bn * npad;
#pragma unroll
      for (int k = 0; k < NPT; ++k) {
        const int p = tid + k * BT;
        if (p < M.n_nodes) {
          cp_async8(un + p, ug + p);
          if (rk[k] >= 0) cp_async8(ln + p, xg + rk[k]);
        }
      }
    }
    double gsum = 0.0, dummy = 0.0;
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
      const int e = tid + k * BT;
      if (e < M.n_el) {
        const int n0 = e01[k] & 0xffffu, n1 = e01[k] >> 16, n2 = e2[k];
        const double l0 = lam[n0], l1 = lam[n1], l2 = lam[n2];
        const double u0 = u[n0], u1 = u[n1], u2 = u[n2];
        st[st_slot(e, half)] = w9[k] * ((l0 + l1) + l2);
        const double g = fma(k12[k] * (l1 - l2), u1 - u2, fma(k02[k] * (l0 - l2), u0 - u2, k01[k] * (l0 - l1) * (u0 - u1)));
        if (gk_per_elem) gk[b * M.n_el + e] = g;
        else gsum += g;
      }
    }
    if (!gk_per_elem) {
      block_sum2(gsum, dummy, sred, lane, warp);   // (contains the barrier that completes st)
      if (tid == 0) gk[b] = gsum;
    } else {
      __syncthreads();
    }
    if (gf) {
#pragma unroll
      for (int k = 0; k < NPT; ++k) {
        const int p = tid + k * BT;
        if (p < M.n_nodes) {
          double g = 0.0;
#pragma unroll
          for (int j = 0; j < 3; ++j) g += st[na[k][j] & 0xffffu] + st[na[k][j] >> 16];
          gf[b * ldgf + p] = g;
        }
      }
    }
    cp_async_wait_all();
    __syncthreads();
    cur ^= 1;
  }
}

int band_npad(const dfe_mesh* m);
// ---------------------------------------------------------------------------------------------------------------------
// Stencil form of the same two kernels for a SCALAR shared kappa (config 5b's own mode): no per-sample CTA barrier at all.
//   forward   F = M_F f with (M_F)_pq = sum_{e∋p,q} area_e / 9 — the load vector of solver.py:143-145 written as a sparse
//             matrix with the pattern of K (<= 7 entries per row on a rectangle() mesh) — minus a per-row lifting constant.
//             (Not the reference's rounding order: u needs 1e-9, and F only enters through the solve; dfe_assemble keeps
//             the bit-exact F.)
//   adjoint   dL/df = M_F lambda (same matrix: it is symmetric), and, because lambda vanishes on Dirichlet nodes,
//             dL/dkappa = -lambda^T K^0 u = -sum_p lambda_p (K^0 u)_p with K^0 the matrix at kappa = 1.
// A thread owns the same SR rows for the whole batch with the row's weights and columns in registers; the rows of f / u /
// lambda are read straight from global memory (each value is used by the 7 rows around it: L1), a CTA loops over samples,
// and the only cross-thread step is a warp-shuffle sum of the dL/dkappa partials (fixed order: k_band_gksum adds the
// per-warp partials of a sample in warp order).
constexpr int SW = 7;          // entries per row
constexpr int SR = 2;          // rows per thread
constexpr int SBT_MAX = 640;   // threads per CTA (=> n_nodes <= 1280)

// ELL tables, one thread per node p: row p of K^0 and of M_F on the full pattern (column-major [j][nnp]), the columns as
// node ids and as free ranks, M_F with the Dirichlet columns zeroed (applied to lambda in free numbering)
__global__ void k_band_ell(const MeshDev M, int nnp, double* __restrict__ ellK, double* __restrict__ ellM,
                           double* __restrict__ ellMr, unsigned* __restrict__ ellc) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_nodes) return;
  double wk[SW], wm[SW];
#pragma unroll
  for (int j = 0; j < SW; ++j) wk[j] = wm[j] = 0.0;
  const int r0 = M.rowptr[p], cnt = M.rowptr[p + 1] - r0;
  for (int a = M.adj_ptr[p]; a < M.adj_ptr[p + 1]; ++a) {
    int nd[3];
    const Elem2D E = elem2d(M, M.adj_elem[a], nd);
    if (E.area < AREA_EPS) continue;
    const int loc = M.adj_loc[a];
    const double den = 4.0 * E.area, w9 = E.area / 9.0;
    for (int q = 0; q < 3; ++q) {
      const int j = M.adj_slot[3 * a + q] - r0;
      const double kv = (E.b[loc] * E.b[q] + E.c[loc] * E.c[q]) / den;
#pragma unroll
      for (int t = 0; t < SW; ++t)
        if (t == j) { wk[t] += kv; wm[t] += w9; }
    }
  }
#pragma unroll
  for (int j = 0; j < SW; ++j) {
    const int c = j < cnt ? M.col[r0 + j] : p;
    const int rk = M.free_rank[c];
    ellK[static_cast<size_t>(j) * nnp + p] = j < cnt ? wk[j] : 0.0;
    ellM[static_cast<size_t>(j) * nnp + p] = j < cnt ? wm[j] : 0.0;
    ellMr[static_cast<size_t>(j) * nnp + p] = (j < cnt && rk >= 0) ? wm[j] : 0.0;
    ellc[static_cast<size_t>(j) * nnp + p] = static_cast<unsigned>(c) | (static_cast<unsigned>(rk >= 0 ? rk : 0) << 16);
  }
}
// liftc[r] = sum_t K[r, d_t] g_t (solver.py:166-169 summed once: it does not depend on the sample)
__global__ void k_band_liftc(const MeshDev M, int npad, const double* __restrict__ liftp, double* __restrict__ liftc) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= npad) return;
  double a = 0.0;
  if (r < M.n_free)
    for (int t = M.lift_ptr[r]; t < M.lift_ptr[r + 1]; ++t) a += liftp[t];
  liftc[r] = a;
}

// The rows of the batch stream through an NST-deep ring in shared memory (cp.async, 8 bytes per element: row starts are
// only 8-byte aligned when n_nodes is odd).  Depth matters more than anything else here: with one row in flight per CTA
// these kernels ran at the latency of a DRAM access per sample (measured 1.05 ms for 1.07 GB); ~64 KB in flight per SM
// are needed to cover it.
constexpr int NST_F = 8, NST_G = 6;
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async8_u32(uint32_t dst, const double* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16_u32(uint32_t dst, const double* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gsrc) : "memory");
}
// Copy the n doubles at src (8-byte aligned) to shared memory so that element p lands at dst16 + 8 * (mis + p), where
// mis = 0 / 1 is the 16-byte phase of src and dst16 is 16-byte aligned: one 8-byte head / tail, 16-byte pairs between.
// Thread 0 issues both: it exists in every CTA, one-warp CTAs included (npad <= 64 / n_nodes <= 64).  (Giving the tail to
// thread 32 instead left it uncopied in a one-warp CTA; thread nt - 1 or a thread of the second warp costs k_band_rhs_fwd3
// up to 10 registers more.)
// Returns mis (the reader's row starts at element `mis` of the stage).
__device__ __forceinline__ int row_to_smem(uint32_t dst16, const double* src, int n, int tid, int nt) {
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(src) >> 3) & 1);
  const int npair = (n - mis) >> 1;
  const double* s2 = src + mis;
  const uint32_t d2 = dst16 + 16u * mis;
  for (int q = tid; q < npair; q += nt) cp_async16_u32(d2 + 16u * q, s2 + 2 * q);
  if (tid == 0 && mis) cp_async8_u32(dst16 + 8u, src);
  if (tid == 0 && ((n - mis) & 1)) cp_async8_u32(dst16 + 8u * (mis + n - 1), src + n - 1);
  return mis;
}

// SPI samples per CTA barrier: with one sample per barrier the loop ran at ~3800 cycles per sample and SM against ~500 issue
// cycles of work (barrier + cp.async issue + shared-memory latency + the dependent fma chain, all exposed); SPI independent
// samples share one barrier and interleave their chains.  The ring holds NG groups of SPI rows.
template <int SPI, int NG>
__global__ void __launch_bounds__(512) k_band_rhs_fwd3(const MeshDev M, long long B, int npad, int nnp,
                                                       const double* __restrict__ f, long long ldf,
                                                       const double* __restrict__ ellM, const unsigned* __restrict__ ellc,
                                                       const double* __restrict__ liftc, double* __restrict__ X) {
  extern __shared__ __align__(16) double sg[];   // [NG][SPI][nnp + 2]
  const int tid = threadIdx.x, nt = blockDim.x;
  double w[SR][SW], lc[SR];
  int c[SR][SW];
#pragma unroll
  for (int k = 0; k < SR; ++k) {
    const int r = tid + k * nt;
    const int p = r < M.n_free ? M.free_nodes[r] : -1;
    lc[k] = r < npad ? liftc[r] : 0.0;
#pragma unroll
    for (int j = 0; j < SW; ++j) {
      w[k][j] = p >= 0 ? ellM[static_cast<size_t>(j) * nnp + p] : 0.0;
      c[k][j] = p >= 0 ? static_cast<int>(ellc[static_cast<size_t>(j) * nnp + p] & 0xffffu) : 0;
    }
  }
  const long long b0 = blockIdx.x, bs = gridDim.x;
  const int pitch = nnp + 2;                          // (room for the 16-byte phase of a row)
  const uint32_t sg32 = smem_u32(sg);
  int st_in = 0;                                      // group slot the next rows go to
  long long b_in = b0;                                // ... and the first sample of that group
  auto issue = [&]() {
#pragma unroll
    for (int s = 0; s < SPI; ++s)
      if (b_in + s * bs < B) row_to_smem(sg32 + 8u * ((st_in * SPI + s) * pitch), f + (b_in + s * bs) * ldf, M.n_nodes, tid, nt);
    cp_async_commit();
    b_in += SPI * bs;
    st_in = st_in + 1 == NG ? 0 : st_in + 1;
  };
  for (int i = 0; i < NG - 1; ++i) issue();
  int st = 0;
  for (long long b = b0; b < B; b += SPI * bs) {
    cp_async_wait<NG - 2>();
    __syncthreads();               // every thread's part of this group has landed, and everybody is done with the previous one
    issue();
#pragma unroll
    for (int k = 0; k < SR; ++k) {
      const int r = tid + k * nt;
      double a[SPI];
#pragma unroll
      for (int s = 0; s < SPI; ++s) {
        const long long bb = b + s * bs;
        const double* fb = sg + (st * SPI + s) * pitch + ((reinterpret_cast<uintptr_t>(f + bb * ldf) >> 3) & 1);
        double v[SW];
#pragma unroll
        for (int j = 0; j < SW; ++j) v[j] = fb[c[k][j]];
        a[s] = -lc[k];
#pragma unroll
        for (int j = 0; j < SW; ++j) a[s] = fma(w[k][j], v[j], a[s]);
      }
#pragma unroll
      for (int s = 0; s < SPI; ++s)
        if (r < npad && b + s * bs < B) X[(b + s * bs) * npad + r] = a[s];
    }
    st = st + 1 == NG ? 0 : st + 1;
  }
  cp_async_wait<0>();
}

// Per-warp partials of lambda^T K^0 u (streams the u and lambda rows) and, with GF, dL/df = M_F lambda in the same pass.
// With GF the kernel costs 96 registers at 576 threads (one CTA per SM, 0.86 ms at config 5b); as two kernels each half
// kept the weights of ONE stencil in registers and two CTAs fit an SM, but the lambda rows were streamed twice
// (0.54 + 0.39 ms).  An adjoint without dL/df launches it without GF.
template <bool GF, int SPI, int NG>
__global__ void __launch_bounds__(SBT_MAX, GF ? 1 : 2) k_band_grad3(const MeshDev M, long long B, int npad, int nnp,
                                                        const double* __restrict__ X, const double* __restrict__ ufull,
                                                        long long ldu, const double* __restrict__ ellK,
                                                        const double* __restrict__ ellMr, const unsigned* __restrict__ ellc,
                                                        double* __restrict__ gkpart, double* __restrict__ gf, long long ldgf) {
  extern __shared__ __align__(16) double sg[];   // [NG][SPI][(nnp + 2) + npad]: u row, lambda row (free numbering)
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int uoff = nnp + 2;                // u row (with room for its 16-byte phase) | lambda row
  const int pitch = uoff + npad;
  double wk[SR][SW], wm[SR][SW];
  unsigned c[SR][SW];
  int rk[SR];
#pragma unroll
  for (int k = 0; k < SR; ++k) {
    const int p = tid + k * nt;
    const bool ex = p < M.n_nodes;
    rk[k] = ex ? M.free_rank[p] : -1;
#pragma unroll
    for (int j = 0; j < SW; ++j) {
      wk[k][j] = ex ? ellK[static_cast<size_t>(j) * nnp + p] : 0.0;
      wm[k][j] = (GF && ex) ? ellMr[static_cast<size_t>(j) * nnp + p] : 0.0;
      c[k][j] = ex ? ellc[static_cast<size_t>(j) * nnp + p] : 0u;
    }
  }
  const long long b0 = blockIdx.x, bs = gridDim.x;
  const uint32_t sg32 = smem_u32(sg);
  int st_in = 0;
  long long b_in = b0;
  auto issue = [&]() {
#pragma unroll
    for (int s = 0; s < SPI; ++s) {
      const long long bb = b_in + s * bs;
      if (bb < B) {
        const uint32_t du = sg32 + 8u * ((st_in * SPI + s) * pitch);
        row_to_smem(du, ufull + bb * ldu, M.n_nodes, tid, nt);
        const double* sl = X + bb * npad;      // 16-byte aligned rows (npad is a multiple of 32)
        for (int q = tid; q < (npad >> 1); q += nt) cp_async16_u32(du + 8u * uoff + 16u * q, sl + 2 * q);
      }
    }
    cp_async_commit();
    b_in += SPI * bs;
    st_in = st_in + 1 == NG ? 0 : st_in + 1;
  };
  for (int i = 0; i < NG - 1; ++i) issue();
  int st = 0;
  for (long long b = b0; b < B; b += SPI * bs) {
    cp_async_wait<NG - 2>();
    __syncthreads();
    issue();
    double part[SPI];
#pragma unroll
    for (int s = 0; s < SPI; ++s) part[s] = 0.0;
#pragma unroll
    for (int k = 0; k < SR; ++k) {
      const int p = tid + k * nt;
#pragma unroll
      for (int s = 0; s < SPI; ++s) {
        const long long bb = b + s * bs;
        const double* ub = sg + (st * SPI + s) * pitch + ((reinterpret_cast<uintptr_t>(ufull + bb * ldu) >> 3) & 1);
        const double* lb = sg + (st * SPI + s) * pitch + uoff;
        double uv[SW];
#pragma unroll
        for (int j = 0; j < SW; ++j) uv[j] = ub[c[k][j] & 0xffffu];
        const double lam = rk[k] >= 0 ? lb[rk[k]] : 0.0;
        double ku = 0.0;
#pragma unroll
        for (int j = 0; j < SW; ++j) ku = fma(wk[k][j], uv[j], ku);
        part[s] = fma(lam, ku, part[s]);
        if (GF) {
          double lv[SW];
#pragma unroll
          for (int j = 0; j < SW; ++j) lv[j] = lb[c[k][j] >> 16];
          double ml = 0.0;
#pragma unroll
          for (int j = 0; j < SW; ++j) ml = fma(wm[k][j], lv[j], ml);
          if (p < M.n_nodes && bb < B) gf[bb * ldgf + p] = ml;
        }
      }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1)
#pragma unroll
      for (int s = 0; s < SPI; ++s) part[s] += __shfl_xor_sync(0xffffffffu, part[s], d);
    if (lane == 0)
#pragma unroll
      for (int s = 0; s < SPI; ++s)
        if (b + s * bs < B) gkpart[(b + s * bs) * nw + warp] = part[s];
    st = st + 1 == NG ? 0 : st + 1;
  }
  cp_async_wait<0>();
}
// dL/dkappa of sample b = -(sum of its per-warp partials, in warp order)
__global__ void k_band_gksum(long long B, int nw, const double* __restrict__ gkpart, double* __restrict__ gk) {
  const long long b = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (b >= B) return;
  double a = 0.0;
  for (int w = 0; w < nw; ++w) a += gkpart[b * nw + w];
  gk[b] = -a;
}

bool band_stencil_fits(const dfe_mesh* m) {
  return m->dev.dim == 2 && m->info.max_row_nnz <= SW && m->dev.n_nodes <= SR * SBT_MAX && m->dev.n_nodes < 65536 &&
         band_npad(m) <= SR * 512 && static_cast<size_t>(NST_G) * (2 * m->dev.n_nodes + 34) * sizeof(double) <= 200 * 1024;
}

// samples per CTA barrier of the stencil-form kernels: the largest of 4 / 2 / 1 whose ring (3 groups for 4, 4 for 2, the
// round-1 depth for 1) fits `row_bytes * rows <= 216 KB`; DFE_BAND_SPI overrides (A/B switch)
int band_spi(size_t row_bytes) {
  const char* e = getenv("DFE_BAND_SPI");   // read per call: the tests compare the variants bit for bit in one process
  const int forced = e ? atoi(e) : 0;
  const size_t cap = 216 * 1024;
  int spi = 12 * row_bytes <= cap ? 4 : 8 * row_bytes <= cap ? 2 : 1;
  if ((forced == 1 || forced == 2 || forced == 4) && forced <= spi) spi = forced;
  return spi;
}

bool band_reg_fits(const dfe_mesh* m) {
  return m->dev.dim == 2 && m->dev.n_el <= EPT * BT && m->dev.n_free <= RPT * BT && m->dev.n_nodes <= NPT * BT &&
         m->dev.n_nodes < 65536 && m->dev.n_el < 65536 && m->n_adj < (1 << 24) && m->n_lift < (1 << 24) &&
         m->dev.n_nodes > 0 && m->n_lift <= 8192 && m->max_adj <= ADJ6;
}

// ---------------------------------------------------------------------------------------------------------------------
// The two triangular solves as a BLOCK-banded TRSM on the FP64 tensor cores (the block-row step and the fragment layout
// are in dfe_band_mma.cuh): two TRIANGULAR 32 x 32 products per block row and right-hand side instead of 32 dependent
// shuffle / fma steps (~2 TFLOP/s: every step waits for the previous one), i.e. a contraction: the one place of this library
// where tensor cores apply.  k_band_blocks builds H once per factorisation (one CTA per block row) and stores H, -S and
// their transposes in the register layout of the DMMA B operand.  (Round 2 first used y_k = H_k b_k + G_k y_{k-1} with the
// full block G_k = -H_k S_k: 26 non-zero 8 x 8 tiles per block row; the two triangular factors have 20, and the kernel is
// bound by the FP64 MMA pipe.)
constexpr int MMA_W = 8;      // warps per CTA of the solve kernel

__global__ void __launch_bounds__(256) k_band_blocks(int npad, const double* __restrict__ invd, const double* __restrict__ Lr,
                                                     double* __restrict__ Ff, double* __restrict__ Bf) {
  __shared__ double D[32][33], S[32][33], U[32][33], H[32][33];
  const int k = blockIdx.x, nb = npad >> 5, tid = threadIdx.x;
  for (int q = tid; q < 1024; q += 256) {
    const int a = q >> 5, b = q & 31;
    const size_t i = static_cast<size_t>(32 * k + a);
    // Lr[i * 32 + d - 1] = L[i][i - d], d = 1..32
    D[a][b] = b < a ? Lr[i * BW + (a - b) - 1] : (a == b ? 1.0 / invd[i] : 0.0);
    S[a][b] = (k > 0 && a <= b) ? Lr[i * BW + (32 + a - b) - 1] : 0.0;                      // L[32k+a][32(k-1)+b]
    U[a][b] = (k + 1 < nb && a <= b) ? Lr[(i + 32) * BW + (32 + a - b) - 1] : 0.0;           // L[32(k+1)+a][32k+b]
    H[a][b] = 0.0;
  }
  __syncthreads();
  if (tid < 32) {   // column tid of H = L_kk^{-1} by forward substitution (pivots 1 / L_ii)
    const int c = tid;
    double h[32];
#pragma unroll
    for (int r = 0; r < 32; ++r) h[r] = 0.0;
#pragma unroll
    for (int r = 0; r < 32; ++r) {
      if (r == c) h[r] = invd[32 * k + r];
      else if (r > c) {
        double sum = 0.0;
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j >= c && j < r) sum = fma(D[r][j], h[j], sum);
        h[r] = -sum * invd[32 * k + r];
      }
    }
#pragma unroll
    for (int r = 0; r < 32; ++r) H[r][c] = h[r];
  }
  __syncthreads();
  double* ff = Ff + static_cast<size_t>(k) * FRAGD;
  double* bf = Bf + static_cast<size_t>(k) * FRAGD;
  for (int q = tid; q < 1024; q += 256) {
    int rr, cc;
    frag_rc(q, rr, cc);
    ff[q] = H[rr][cc];            // forward:  out[s][r] += in[s][c] H[r][c]          (zero for c > r)
    ff[1024 + q] = -S[rr][cc];    //           t[s][r]   += y_prev[s][c] (-S[r][c])    (zero for c < r)
    bf[q] = H[cc][rr];            // backward: out[s][r] += in[s][c] H[c][r]          (zero for c < r)
    bf[1024 + q] = -U[cc][rr];    //           t[s][r]   += x_next[s][c] (-U[c][r])    (zero for c > r)
  }
}

// GIN: the right-hand sides are gathered from a (B, n_nodes) array in node numbering (gsrc[b * ldg + free_nodes[r]], the
// adjoint's gbar restricted to the free rows) instead of being read from X; SOUT: the solution is scattered straight into
// u (u[b * ldu + free_nodes[r]], solver.py:177-181, with the Dirichlet values) instead of being written back to X.  Either
// saves a pass over the batch (0.25 + 0.27 ms of pure copies at config 5b); X still holds y between the passes.
template <bool GIN, bool SOUT>
__global__ void __launch_bounds__(32 * MMA_W, 2) k_band_solve_mma(int npad, long long B, const double* __restrict__ Ff,
                                                                  const double* __restrict__ Bf, double* __restrict__ X,
                                                                  const int* __restrict__ fnode, int nfree,
                                                                  const double* __restrict__ gsrc, long long ldg,
                                                                  double* __restrict__ uout, long long ldu,
                                                                  const int* __restrict__ dir_idx,
                                                                  const double* __restrict__ dir_val, int n_dir) {
  __shared__ __align__(16) double stg[2][FRAGD];
  __shared__ uint64_t bar[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, q = lane & 3;
  const int nb = npad >> 5, nsteps = 2 * nb;
  const long long s0 = (blockIdx.x * static_cast<long long>(MMA_W) + warp) * MMA_S;
  double* row[2];
  const double* grow[2];
  double* urow[2];
  bool valid[2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const long long sidx = s0 + 8 * mt + g;
    valid[mt] = sidx < B;
    const long long sc = valid[mt] ? sidx : B - 1;
    row[mt] = X + sc * npad + 2 * q;
    grow[mt] = GIN ? gsrc + sc * ldg : nullptr;
    urow[mt] = SOUT ? uout + sc * ldu : nullptr;
  }
  // right-hand side of block row kb: from X, or gathered through the free-node table
  auto load_rhs = [&](int kb, Blk& Rr) {
    if (!GIN) {
      ld_block(row, kb, Rr);
    } else {
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int c0 = 32 * kb + 8 * nt + 2 * q;
        const int n0 = c0 < nfree ? fnode[c0] : -1, n1 = c0 + 1 < nfree ? fnode[c0 + 1] : -1;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          Rr[mt][nt][0] = n0 >= 0 ? grow[mt][n0] : 0.0;
          Rr[mt][nt][1] = n1 >= 0 ? grow[mt][n1] : 0.0;
        }
      }
    }
  };
  if (tid == 0) {
    mbar_init_raw(&bar[0], 1);
    mbar_init_raw(&bar[1], 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(&bar[0], FRAGD * 8u);
    bulk_g2s(stg[0], frag_src(Ff, Bf, nb, 0), FRAGD * 8u, &bar[0]);
  }
  Blk R, P = {}, acc;
  load_rhs(0, R);
  for (int step = 0; step < nsteps; ++step) {
    const int k = band_block(step, nb);
    __syncthreads();   // every warp has finished step - 1: the other stage is free (and, at step 0, the barriers exist)
    if (tid == 0 && step + 1 < nsteps) {
      mbar_arrive_expect_tx(&bar[(step + 1) & 1], FRAGD * 8u);
      bulk_g2s(stg[(step + 1) & 1], frag_src(Ff, Bf, nb, step + 1), FRAGD * 8u, &bar[(step + 1) & 1]);
    }
    mbar_wait(&bar[step & 1], (step >> 1) & 1);
    Blk t;
    blk_copy(t, R);
    const int knext = band_block(step + 1, nb);   // == k at the turn-around
    // the right-hand side of the next step is in flight while the two products run: the next block of b (forward pass)
    // or of y (backward pass)
    if (step + 1 < nsteps && knext != k) {
      if (GIN && step + 1 < nb) load_rhs(knext, R);
      else ld_block(row, knext, R);
    }
    band_step(step, nb, stg[step & 1], lane, t, P, acc);
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        P[mt][nt][0] = acc[mt][nt][0];
        P[mt][nt][1] = acc[mt][nt][1];
        if (knext == k) { R[mt][nt][0] = acc[mt][nt][0]; R[mt][nt][1] = acc[mt][nt][1]; }   // turn-around: y_{nb-1} is the next rhs
        if (SOUT && step >= nb) {          // backward pass: x_k is final — straight into u
          const int c0 = 32 * k + 8 * nt + 2 * q;
          if (valid[mt] && c0 < nfree) urow[mt][fnode[c0]] = acc[mt][nt][0];
          if (valid[mt] && c0 + 1 < nfree) urow[mt][fnode[c0 + 1]] = acc[mt][nt][1];
        } else if (valid[mt]) {
          *reinterpret_cast<double2*>(row[mt] + 32 * k + 8 * nt) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);
        }
      }
  }
  if (SOUT && n_dir > 0) {   // u[d] = g on the Dirichlet nodes of the warp's samples (solver.py:177-179): scattered 8-byte
    // stores that hide behind the other warps' MMAs here; as a kernel of their own they cost 68 us at config 5b
    for (int d = lane; d < n_dir; d += 32) {
      const int node = dir_idx[d];
      const double gv = dir_val[d];
      for (int sidx = 0; sidx < MMA_S; ++sidx)
        if (s0 + sidx < B) uout[(s0 + sidx) * ldu + node] = gv;
    }
  }
}

// adjoint: dL/dkappa (per element, or summed per sample in a fixed order) and dL/df from lambda = X (0 on Dirichlet
// nodes).  One CTA per sample: lambda on all nodes and the per-element sums lambda_i+lambda_j+lambda_k in shared memory.
__global__ void __launch_bounds__(BT) k_band_grad(const MeshDev M, long long B, int npad, const double* __restrict__ X,
                                                  const double* __restrict__ ufull, long long ldu,
                                                  const double* __restrict__ geom, double* __restrict__ gk,
                                                  int gk_per_elem, double* __restrict__ gf, long long ldgf) {
  extern __shared__ double sg[];
  double* slam = sg;                 // [n_nodes]
  double* su = slam + M.n_nodes;     // [n_nodes]
  double* ssum = su + M.n_nodes;     // [n_el]
  double* sred = ssum + M.n_el;      // [2 * BNW]
  const size_t ne = static_cast<size_t>(M.n_el);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (long long b = blockIdx.x; b < B; b += gridDim.x) {
    const double* lamf = X + b * npad;
    const double* ug = ufull + b * ldu;
    for (int p = tid; p < M.n_nodes; p += BT) {
      const int rk = M.free_rank[p];
      slam[p] = rk >= 0 ? lamf[rk] : 0.0;
      su[p] = ug[p];
    }
    const double* u = su;
    __syncthreads();
    double gsum = 0.0, dummy = 0.0;
    for (int e = tid; e < M.n_el; e += BT) {
      double ge[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) ge[k] = (k == 1) ? 0.0 : geom[k * ne + e];
      double g = 0.0;
      if (M.dim == 1) {
        const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
        g = -(slam[j] - slam[i]) * (u[j] - u[i]) / ge[2];
      } else {
        const int n0 = M.elems[3 * e], n1 = M.elems[3 * e + 1], n2 = M.elems[3 * e + 2];
        const double l0 = slam[n0], l1 = slam[n1], l2 = slam[n2];
        ssum[e] = (l0 + l1) + l2;
        if (ge[0] >= 0.0) {
          const double u0 = u[n0], u1 = u[n1], u2 = u[n2];
          const double bl = fma(ge[4], l2, fma(ge[3], l1, fma(ge[2], l0, 0.0)));
          const double bu = fma(ge[4], u2, fma(ge[3], u1, fma(ge[2], u0, 0.0)));
          const double cl = fma(ge[7], l2, fma(ge[6], l1, fma(ge[5], l0, 0.0)));
          const double cu = fma(ge[7], u2, fma(ge[6], u1, fma(ge[5], u0, 0.0)));
          g = -(bl * bu + cl * cu) / (12.0 * ge[0]);   // 4 area = 12 (area/3)
        }
      }
      if (gk_per_elem) gk[b * M.n_el + e] = g;
      else gsum += g;
    }
    if (!gk_per_elem) {
      block_sum2(gsum, dummy, sred, lane, warp);
      if (tid == 0) gk[b] = gsum;
    }
    __syncthreads();   // ssum complete
    if (gf) {
      for (int pn = tid; pn < M.n_nodes; pn += BT) {
        double g = 0.0;
        for (int a = M.adj_ptr[pn]; a < M.adj_ptr[pn + 1]; ++a) {
          const int e = M.adj_elem[a];
          const double w9 = geom[ne + e];
          if (M.dim == 1) g = fma(w9, slam[pn], g);
          else if (w9 >= 0.0) g = fma(w9, ssum[e], g);
        }
        gf[b * ldgf + pn] = g;
      }
    }
    __syncthreads();   // slam / ssum are reused by the next sample
  }
}

int band_width(const dfe_mesh* m) {   // max |row - col| over the pattern of K_free
  long long w = 0;
  const long long n = static_cast<long long>(m->h_rowptr_f.size()) - 1;
  for (long long r = 0; r < n; ++r)
    for (long long k = m->h_rowptr_f[r]; k < m->h_rowptr_f[r + 1]; ++k) {
      const long long d = r > m->h_col_f[k] ? r - m->h_col_f[k] : m->h_col_f[k] - r;
      if (d > w) w = d;
    }
  return static_cast<int>(w);
}
bool band_fits(const dfe_mesh* m) {
  if (!m || m->info.device < 0 || m->dev.n_free < 1 || m->dev.npe != m->dev.dim + 1) return false;   // P1 load / gradient kernels
  // the gradient kernel keeps lambda (all nodes) and one sum per element in shared memory
  if ((2 * static_cast<size_t>(m->dev.n_nodes) + m->dev.n_el + 2 * BNW) * sizeof(double) > 200 * 1024) return false;
  return band_width(m) <= BW;
}
int band_npad(const dfe_mesh* m) { return ((m->dev.n_free + 31) / 32) * 32; }

size_t batch_smem(const dfe_mesh* m, bool bwd) {
  const size_t snz = static_cast<size_t>(m->dev.sell_nnz);
  size_t d = snz + 32ull * m->dev.n_slices + 6 * BNW + (bwd ? static_cast<size_t>(m->dev.n_nodes) : 0);
  return d * sizeof(double) + snz * sizeof(int) + 16;
}

bool batch_fits(const dfe_mesh* m) {
  if (!m || m->info.device < 0 || m->dev.n_free < 1 || m->dev.npe != m->dev.dim + 1) return false;   // P1 load / gradient kernels
  if (m->dev.n_slices > BNW * RPT_MAX) return false;
  return batch_smem(m, true) <= 200 * 1024;
}

template <bool BWD, int RPT>
int launch(const dfe_mesh* m, const BArgs& A, cudaStream_t st) {
  auto kern = k_batch<BWD, RPT>;
  const size_t smem = batch_smem(m, BWD);
  DFE_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int occ = 0;
  DFE_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, BT, smem));
  if (occ < 1) {
    dfe::set_error("dfe_batch: kernel does not fit (shared memory %zu bytes)", smem);
    return DFE_ERR_UNSUPPORTED;
  }
  long long grid = static_cast<long long>(occ) * m->sm_count;
  if (grid > A.B) grid = A.B;
  kern<<<static_cast<unsigned>(grid), BT, smem, st>>>(A);
  DFE_CUDA_OK(cudaGetLastError());
  return DFE_OK;
}

template <bool BWD>
int dispatch(const dfe_mesh* m, const BArgs& A, cudaStream_t st) {
  const int rpt = (m->dev.n_slices + BNW - 1) / BNW;
  switch (rpt) {
    case 1: return launch<BWD, 1>(m, A, st);
    case 2: return launch<BWD, 2>(m, A, st);
    case 3: return launch<BWD, 3>(m, A, st);
    case 4: return launch<BWD, 4>(m, A, st);
    case 5: case 6: return launch<BWD, 6>(m, A, st);
    default: return launch<BWD, 8>(m, A, st);
  }
}

int enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (!batch_fits(m)) {
    dfe::set_error("%s: mesh too large for the shared-memory resident batched solver (n_free %lld > %d or matrix > 200 KB); "
                   "use dfe_assemble / dfe_eliminate / dfe_pcg per sample", who, static_cast<long long>(m->info.n_free),
                   32 * BNW * RPT_MAX);
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}

}  // namespace

extern "C" int dfe_batch_supported(const dfe_mesh* m) { return batch_fits(m) ? 1 : 0; }

extern "C" int dfe_batch_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* vals_full,
                             const double* sell_vals, const double* dinv, double* u, int64_t ldu, double tol,
                             int64_t maxit, int32_t* iters, double* relres, int32_t* status, void* stream) {
  int prev;
  int rc = enter(m, "dfe_batch_fwd", &prev);
  if (rc) return rc;
  if (!f || !vals_full || !sell_vals || !dinv || !u || !iters || !relres || !status || B < 1 || !(tol > 0.0) || maxit < 1) {
    dfe::set_error("dfe_batch_fwd: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else {
    BArgs A{};
    A.M = m->dev; A.B = B; A.in = f; A.ldin = ldf; A.vals_full = vals_full; A.sell_vals = sell_vals; A.dinv = dinv;
    A.out = u; A.ldout = ldu; A.tol = tol; A.maxit = static_cast<int>(maxit > 2000000000 ? 2000000000 : maxit);
    A.iters = iters; A.relres = relres; A.status = status;
    rc = dispatch<false>(m, A, static_cast<cudaStream_t>(stream));
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_batch_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                             const double* sell_vals, const double* dinv, int kappa_mode, double* gf, int64_t ldgf,
                             double* gkappa, double tol, int64_t maxit, int32_t* iters, double* relres, int32_t* status,
                             void* stream) {
  int prev;
  int rc = enter(m, "dfe_batch_bwd", &prev);
  if (rc) return rc;
  if (!gbar || !u || !sell_vals || !dinv || !gkappa || !iters || !relres || !status || B < 1 || !(tol > 0.0) || maxit < 1) {
    dfe::set_error("dfe_batch_bwd: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_SCALAR && kappa_mode != DFE_KAPPA_PER_ELEMENT) {
    dfe::set_error("dfe_batch_bwd: kappa_mode must be SCALAR or PER_ELEMENT (the batch shares one matrix)");
    rc = DFE_ERR_INVALID;
  } else {
    BArgs A{};
    A.M = m->dev; A.B = B; A.in = gbar; A.ldin = ldg; A.u = u; A.ldu = ldu; A.sell_vals = sell_vals; A.dinv = dinv;
    A.out = gf; A.ldout = ldgf; A.gk = gkappa; A.gk_per_elem = kappa_mode == DFE_KAPPA_PER_ELEMENT;
    A.tol = tol; A.maxit = static_cast<int>(maxit > 2000000000 ? 2000000000 : maxit);
    A.iters = iters; A.relres = relres; A.status = status;
    rc = dispatch<true>(m, A, static_cast<cudaStream_t>(stream));
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

// ---------------------------------------------------------------------------------------------- banded direct ABI
extern "C" int dfe_band_supported(const dfe_mesh* m) { return band_fits(m) ? 1 : 0; }

extern "C" size_t dfe_band_factor_bytes(const dfe_mesh* m) {
  if (!m) return 0;
  const size_t np = static_cast<size_t>(band_npad(m));
  const size_t nnp = (static_cast<size_t>(m->dev.n_nodes) + 1) & ~static_cast<size_t>(1);
  return (np + np * BW + 12 * static_cast<size_t>(m->dev.n_el) + static_cast<size_t>(m->n_lift) + (np + 40) * (BW + 1) +
          2 * (np / 32) * FRAGD + 8 + (3 * SW + SW / 2 + 1) * nnp + np) * sizeof(double) + 512;
}
extern "C" size_t dfe_band_workspace_bytes(const dfe_mesh* m, int64_t B) {
  if (!m || B < 1) return 0;
  return static_cast<size_t>(B) * (band_npad(m) + 32) * sizeof(double);   // X (B, npad) | per-warp dL/dkappa partials (B, <= 32)
}

namespace {
struct BandPtrs {
  double *invd, *Lr, *geom, *geom2, *liftp, *Ab, *Ff, *Bf, *ellK, *ellM, *ellMr, *liftc;
  unsigned* ellc;
  int nnp;
  int* status;
};
BandPtrs band_ptrs(const dfe_mesh* m, void* factor) {
  const size_t np = static_cast<size_t>(band_npad(m));
  BandPtrs p;
  p.invd = static_cast<double*>(factor);
  p.Lr = p.invd + np;
  p.geom = p.Lr + np * BW;
  p.geom2 = p.geom + 8 * static_cast<size_t>(m->dev.n_el);
  p.liftp = p.geom2 + 4 * static_cast<size_t>(m->dev.n_el);
  p.Ab = p.liftp + m->n_lift;
  p.Ff = p.Ab + (np + 40) * (BW + 1);
  p.Ff += (16 - (reinterpret_cast<uintptr_t>(p.Ff) & 15)) / 8 % 2;   // 16-byte alignment for the bulk copies
  p.Bf = p.Ff + (np / 32) * FRAGD;
  p.nnp = (m->dev.n_nodes + 1) & ~1;
  p.ellK = p.Bf + (np / 32) * FRAGD;
  p.ellM = p.ellK + static_cast<size_t>(SW) * p.nnp;
  p.ellMr = p.ellM + static_cast<size_t>(SW) * p.nnp;
  p.liftc = p.ellMr + static_cast<size_t>(SW) * p.nnp;
  p.ellc = reinterpret_cast<unsigned*>(p.liftc + np);
  p.status = reinterpret_cast<int*>(p.ellc + static_cast<size_t>(SW) * p.nnp + 2);
  return p;
}
int band_enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (!band_fits(m)) {
    dfe::set_error("%s: half bandwidth of K_free is %d > %d; use dfe_batch_* (PCG) or the per-sample path", who, band_width(m), BW);
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}
inline unsigned nblk(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

// L y = b, L^T x = y for the whole batch, in place on X: block TRSM on the FP64 tensor cores
void band_solve(int np, long long B, const BandPtrs& p, double* X, cudaStream_t st) {
  k_band_solve_mma<false, false><<<nblk(B, MMA_W * MMA_S), 32 * MMA_W, 0, st>>>(np, B, p.Ff, p.Bf, X, nullptr, 0, nullptr, 0,
                                                                                nullptr, 0, nullptr, nullptr, 0);
}
}  // namespace

void dfe::band_frags(const dfe_mesh* m, const void* factor, const double** Ff, const double** Bf) {
  const BandPtrs p = band_ptrs(m, const_cast<void*>(factor));
  *Ff = p.Ff;
  *Bf = p.Bf;
}

void dfe::band_tables(const dfe_mesh* m, double* geom, double* geom2, cudaStream_t st) {
  k_band_geom<<<nblk(m->dev.n_el, 128), 128, 0, st>>>(m->dev, geom);
  k_band_tables<<<nblk(m->dev.n_el, 128), 128, 0, st>>>(m->dev, nullptr, 0, nullptr, geom2);
}

void dfe::band_rhs(const dfe_mesh* m, long long B, const double* f, long long ldf, const double* vals_full,
                   long long vstride, const double* geom, double* X, cudaStream_t st) {
  const size_t rsm = (static_cast<size_t>(m->dev.n_nodes) + m->dev.n_el) * sizeof(double);
  cudaFuncSetAttribute(k_band_rhs_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rsm));
  long long rgrid = 8LL * m->sm_count;
  if (rgrid > B) rgrid = B;
  k_band_rhs_fwd<<<static_cast<unsigned>(rgrid), BT, rsm, st>>>(m->dev, B, band_npad(m), f, ldf, vals_full, vstride, geom, X);
}

int dfe::band_grad(const dfe_mesh* m, long long B, const double* X, const double* u, long long ldu, const double* geom,
                   const double* geom2, int gk_per_elem, double* gk, double* gf, long long ldgf, cudaStream_t st) {
  const int np = band_npad(m);
  if (band_reg_fits(m)) {
    const int nnp = (m->dev.n_nodes + 1) & ~1;
    const size_t gsm2 = (4 * static_cast<size_t>(nnp) + m->dev.n_el + 4 + 2 * BNW) * sizeof(double);
    cudaFuncSetAttribute(k_band_grad2, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(gsm2));
    long long grid = 2LL * m->sm_count;
    if (grid > B) grid = B;
    k_band_grad2<<<static_cast<unsigned>(grid), BT, gsm2, st>>>(m->dev, B, np, X, u, ldu, geom2, gk, gk_per_elem, gf, ldgf, nnp);
    return DFE_OK;
  }
  const size_t gsm = (2 * static_cast<size_t>(m->dev.n_nodes) + m->dev.n_el + 2 * BNW) * sizeof(double);
  if (gsm > 200 * 1024) {
    dfe::set_error("banded adjoint: mesh too large for the gradient kernel (%zu bytes of shared memory)", gsm);
    return DFE_ERR_UNSUPPORTED;
  }
  cudaFuncSetAttribute(k_band_grad, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(gsm));
  long long grid = 8LL * m->sm_count;
  if (grid > B) grid = B;
  k_band_grad<<<static_cast<unsigned>(grid), BT, gsm, st>>>(m->dev, B, np, X, u, ldu, geom, gk, gk_per_elem, gf, ldgf);
  return DFE_OK;
}

// K_free = L L^T from the assembled matrix (dfe_assemble); `factor` holds dfe_band_factor_bytes(m) bytes.  The status
// word (0 ok, 5 = a pivot <= 0: K_free is not SPD) is the int at the end of the buffer; *status_dev (optional, device)
// receives a copy.  Asynchronous.
extern "C" int dfe_band_factor(const dfe_mesh* m, const double* vals_full, void* factor, int32_t* status_dev, void* stream) {
  int prev;
  int rc = band_enter(m, "dfe_band_factor", &prev);
  if (rc) return rc;
  if (!vals_full || !factor) {
    dfe::set_error("dfe_band_factor: null argument");
    rc = DFE_ERR_INVALID;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const BandPtrs p = band_ptrs(m, factor);
    const size_t np = static_cast<size_t>(band_npad(m));
    // invd | Lr zeroed (rows >= n_free and entries outside the band stay zero), Ab zeroed, then gathered
    cudaError_t e = cudaMemsetAsync(p.invd, 0, (np + np * BW) * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(p.Ab, 0, (np + 40) * (BW + 1) * sizeof(double), st);
    k_band_gather<<<nblk(m->dev.n_free, 128), 128, 0, st>>>(m->dev, vals_full, p.Ab);
    // (running the Cholesky chain on a second stream under the load-vector kernel of dfe_band_fwd was measured: no gain —
    // the one-CTA factorisation is latency-bound and slows down under a bandwidth-bound neighbour as much as it overlaps)
    k_band_factor_blk<<<1, 256, 0, st>>>(m->dev.n_free, band_npad(m), p.Ab, p.invd, p.Lr, p.status);
    k_band_blocks<<<static_cast<unsigned>(np / 32), 256, 0, st>>>(band_npad(m), p.invd, p.Lr, p.Ff, p.Bf);
    if (e == cudaSuccess && status_dev) e = cudaMemcpyAsync(status_dev, p.status, sizeof(int), cudaMemcpyDeviceToDevice, st);
    k_band_geom<<<nblk(m->dev.n_el, 128), 128, 0, st>>>(m->dev, p.geom);
    {
      const int nt = m->dev.n_el > m->n_lift ? m->dev.n_el : m->n_lift;
      k_band_tables<<<nblk(nt, 128), 128, 0, st>>>(m->dev, vals_full, m->n_lift, p.liftp, p.geom2);
      if (band_stencil_fits(m)) {
        k_band_ell<<<nblk(m->dev.n_nodes, 128), 128, 0, st>>>(m->dev, p.nnp, p.ellK, p.ellM, p.ellMr, p.ellc);
        k_band_liftc<<<nblk(band_npad(m), 128), 128, 0, st>>>(m->dev, band_npad(m), p.liftp, p.liftc);
      }
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
      dfe::set_error("dfe_band_factor: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_band_fwd(const dfe_mesh* m, int64_t B, const double* f, int64_t ldf, const double* vals_full,
                            const void* factor, double* u, int64_t ldu, void* ws, size_t ws_bytes, void* stream) {
  int prev;
  int rc = band_enter(m, "dfe_band_fwd", &prev);
  if (rc) return rc;
  if (!f || !vals_full || !factor || !u || !ws || B < 1 || ldf < m->dev.n_nodes || ldu < m->dev.n_nodes) {
    dfe::set_error("dfe_band_fwd: null / invalid argument (row strides must be >= n_nodes)");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_band_workspace_bytes(m, B)) {
    dfe::set_error("dfe_band_fwd: workspace %zu bytes < required %zu", ws_bytes, dfe_band_workspace_bytes(m, B));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int np = band_npad(m);
    const BandPtrs p = band_ptrs(m, const_cast<void*>(factor));
    double* X = static_cast<double*>(ws);
    if (band_stencil_fits(m)) {
      const int nt = ((np + SR - 1) / SR + 31) & ~31;
      const size_t row = static_cast<size_t>(p.nnp + 2) * sizeof(double);
      auto launch_rhs = [&](auto kern, int rows) {
        const size_t sm3 = rows * row;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm3));
        int occ = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, sm3);
        long long rgrid = static_cast<long long>(occ > 0 ? occ : 1) * m->sm_count;   // persistent: one wave
        if (rgrid > B) rgrid = B;
        kern<<<static_cast<unsigned>(rgrid), nt, sm3, st>>>(m->dev, B, np, p.nnp, f, ldf, p.ellM, p.ellc, p.liftc, X);
      };
      switch (band_spi(row)) {
        case 4: launch_rhs(k_band_rhs_fwd3<4, 3>, 12); break;
        case 2: launch_rhs(k_band_rhs_fwd3<2, 4>, 8); break;
        default: launch_rhs(k_band_rhs_fwd3<1, NST_F>, NST_F); break;
      }
    } else {
      dfe::band_rhs(m, B, f, ldf, vals_full, 0, p.geom, X, st);
    }
    k_band_solve_mma<false, true><<<nblk(B, MMA_W * MMA_S), 32 * MMA_W, 0, st>>>(np, B, p.Ff, p.Bf, X, m->dev.free_nodes,
                                                                                 m->dev.n_free, nullptr, 0, u, ldu,
                                                                                 m->dev.dir_idx, m->dev.dir_val, m->dev.n_dir);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      dfe::set_error("dfe_band_fwd: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_band_bwd(const dfe_mesh* m, int64_t B, const double* gbar, int64_t ldg, const double* u, int64_t ldu,
                            const void* factor, int kappa_mode, double* gf, int64_t ldgf, double* gkappa, void* ws,
                            size_t ws_bytes, void* stream) {
  int prev;
  int rc = band_enter(m, "dfe_band_bwd", &prev);
  if (rc) return rc;
  if (!gbar || !u || !factor || !gkappa || !ws || B < 1 || ldg < m->dev.n_nodes || ldu < m->dev.n_nodes ||
      (gf && ldgf < m->dev.n_nodes)) {
    dfe::set_error("dfe_band_bwd: null / invalid argument (row strides must be >= n_nodes)");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_SCALAR && kappa_mode != DFE_KAPPA_PER_ELEMENT) {
    dfe::set_error("dfe_band_bwd: kappa_mode must be SCALAR or PER_ELEMENT (the batch shares one matrix)");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_band_workspace_bytes(m, B)) {
    dfe::set_error("dfe_band_bwd: workspace %zu bytes < required %zu", ws_bytes, dfe_band_workspace_bytes(m, B));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int np = band_npad(m);
    const BandPtrs p = band_ptrs(m, const_cast<void*>(factor));
    double* X = static_cast<double*>(ws);
    k_band_solve_mma<true, false><<<nblk(B, MMA_W * MMA_S), 32 * MMA_W, 0, st>>>(np, B, p.Ff, p.Bf, X, m->dev.free_nodes,
                                                                                 m->dev.n_free, gbar, ldg, nullptr, 0, nullptr, nullptr, 0);
    if (kappa_mode == DFE_KAPPA_SCALAR && band_stencil_fits(m)) {
      const int nt = ((m->dev.n_nodes + SR - 1) / SR + 31) & ~31;
      double* gkpart = X + static_cast<size_t>(B) * np;
      auto launch_grad = [&](auto kern, size_t sm3, double* gfp) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm3));
        int occ = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, sm3);
        long long grid = static_cast<long long>(occ > 0 ? occ : 1) * m->sm_count;   // persistent: one wave
        if (grid > B) grid = B;
        kern<<<static_cast<unsigned>(grid), nt, sm3, st>>>(m->dev, B, np, p.nnp, X, u, ldu, p.ellK, p.ellMr, p.ellc, gkpart, gfp, ldgf);
      };
      const size_t row = static_cast<size_t>(p.nnp + 2 + np) * sizeof(double);
      if (gf) {
        switch (band_spi(row)) {
          case 4: launch_grad(k_band_grad3<true, 4, 3>, 12 * row, gf); break;
          case 2: launch_grad(k_band_grad3<true, 2, 4>, 8 * row, gf); break;
          default: launch_grad(k_band_grad3<true, 1, NST_G>, NST_G * row, gf); break;
        }
      } else {
        switch (band_spi(2 * row)) {   // two CTAs per SM without dL/df
          case 4: launch_grad(k_band_grad3<false, 4, 3>, 12 * row, nullptr); break;
          case 2: launch_grad(k_band_grad3<false, 2, 4>, 8 * row, nullptr); break;
          default: launch_grad(k_band_grad3<false, 1, NST_G>, NST_G * row, nullptr); break;
        }
      }
      k_band_gksum<<<nblk(B, 256), 256, 0, st>>>(B, nt / 32, gkpart, gkappa);
    } else {
      rc = dfe::band_grad(m, B, X, u, ldu, p.geom, p.geom2, kappa_mode == DFE_KAPPA_PER_ELEMENT, gkappa, gf, ldgf, st);
    }
    cudaError_t e = cudaGetLastError();
    if (rc == DFE_OK && e != cudaSuccess) {
      dfe::set_error("dfe_band_bwd: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int64_t dfe_band_npad(const dfe_mesh* m) { return (m && band_fits(m)) ? band_npad(m) : 0; }

// X <- A_free^{-1} X for B right-hand sides in free numbering, in place (the two triangular solves alone)
extern "C" int dfe_band_solve(const dfe_mesh* m, int64_t B, double* X, const void* factor, void* stream) {
  int prev;
  int rc = band_enter(m, "dfe_band_solve", &prev);
  if (rc) return rc;
  if (!X || !factor || B < 1 || (reinterpret_cast<uintptr_t>(X) & 15)) {
    dfe::set_error("dfe_band_solve: null / invalid argument (X must be 16-byte aligned)");
    rc = DFE_ERR_INVALID;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    band_solve(band_npad(m), B, band_ptrs(m, const_cast<void*>(factor)), X, st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      dfe::set_error("dfe_band_solve: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}
