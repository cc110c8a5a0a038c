// Multigrid-preconditioned conjugate gradients for meshes with the topology of FEMesh.rectangle(), one cooperative
// persistent kernel per solve (sm_100a).
//
// Replaces torch.linalg.solve(K_free, F_free) (diffhe/solver.py:174) and — called with gbar_free — the adjoint solve
// of LinalgSolveExBackward0, like dfe_pcg, for the meshes reference mesh.py:79-121 produces (node id = row*(nx+1)+col,
// triangles [a,b,d], [b,c,d] per quad, all four sides Dirichlet).  Jacobi-PCG needs O(nx) iterations there (7435 at
// 1024 x 1024 with a 1e3 coefficient contrast, SURVEY §7 hard part 2); a V-cycle preconditioner needs ~50.
//
// Structure used.  For right triangles the two acute vertices of an element do not couple (grad phi_b . grad phi_d = 0
// exactly, also in floating point: one factor of each product is an exact 0), so K_free is numerically a 5-point
// operator on the (ny-1) x (nx-1) grid of interior nodes, whatever kappa_e is.  dfe_mg_setup reads the bit-exact
// assembled values (dfe_assemble) into stencil form (centre / east / north; west and south by symmetry — K is
// bitwise symmetric) and verifies that the structural hypotenuse entries are exact zeros (DFE_ERR_UNSUPPORTED
// otherwise: the caller falls back to dfe_pcg).  The outer CG applies exactly this operator.
//
// Preconditioner: V(nu, nu) cycle, damped Jacobi (omega = 0.8; symmetric, so the cycle is an SPD operator and plain
// CG applies), standard coarsening (coarse node (I, J) = fine node (2I+1, 2J+1)), OPERATOR-DEPENDENT interpolation
// (Dendy's black-box multigrid weights from the collapsed stencils — the coefficient jumps by 1e3 from element to
// element, bilinear weights cost 25 % more iterations), Galerkin coarse operators P^T A P (9-point, stored as centre /
// E / N / NE / NW), an explicit inverse on the coarsest grid (<= 32 unknowns).  Built once per matrix by
// dfe_mg_setup and reused by the adjoint solve.
//
// Solve kernel: one 768-thread CTA per SM, every level's nodes split into contiguous per-CTA ranges; the phases of
// the cycle (smooth / residual / restrict / prolong) and of CG (q = A p, vector updates) are separated by the
// fixed-order grid reduction of dfe_gridsync.cuh, which doubles as the barrier: dot products are bit-reproducible,
// no float atomics.  Stops at recursive ||r|| <= tol ||rhs||, on the rhs scaled by the power of two that brings its largest
// entry into [1, 2) (x is scaled back at the end; see k_pcg).
#include <cmath>
#include <cstdlib>
#include <vector>

#include "dfe_internal.h"

namespace {

#include "dfe_gridsync.cuh"

constexpr int MG_MAXL = 12;
constexpr int MG_COARSEST = 32;    // unknowns of the coarsest grid (explicit inverse)
constexpr double OMEGA1 = 0.8;   // one sweep: optimal single damping for the high-frequency range [1/2, 2] of D^-1 A
// Damping of sweep k = 1 .. nu.  One sweep: 0.8.  More: the reciprocals of the roots of the Chebyshev polynomial of degree nu
// on [1/2, 2] — the eigenvalue range of D^-1 A that standard coarsening leaves to the smoother (lambda_max <= 2 by
// Gershgorin for these M-matrices).  Two sweeps then damp the range by 1 / T_2(5/3) = 0.22 instead of 0.6^2 = 0.36; the
// smoother is still a polynomial in D^-1 A, so the V-cycle stays symmetric positive definite.  DFE_MG_CHEB=0: constant 0.8.
inline void mg_omegas(int nu, double* om) {
  static const bool cheb = [] { const char* e = getenv("DFE_MG_CHEB"); return !(e && e[0] == '0'); }();
  for (int k = 0; k < 8; ++k) om[k] = OMEGA1;
  if (!cheb || nu < 2) return;
  const double theta = 1.25, delta = 0.75, pi = 3.14159265358979323846;
  for (int k = 1; k <= nu && k <= 8; ++k) om[k - 1] = 1.0 / (theta + delta * cos((2 * k - 1) * pi / (2.0 * nu)));
}

struct MgMat {   // one level; pointers into the hierarchy buffer
  int my, mx, n, nine;
  double *C, *dinv, *E, *N, *NE, *NW;   // A(i,j)-(i,j+1) = E, -(i+1,j) = N, -(i+1,j+1) = NE, -(i+1,j-1) = NW
  double* pw;                           // [4][n] interpolation weights towards the next coarser level
};
struct MgVec {
  double *b, *r, *xa, *xb;
};
struct MgHier {
  int L, nc;
  MgMat lev[MG_MAXL];
  double* cinv;   // [nc][nc] inverse of the coarsest operator
  int* flag;      // set by k_mg_extract when a structural off-stencil entry is not an exact zero / a pivot is bad
};

// ---------------------------------------------------------------------------------------------- stencil access
// coupling between node (i, j) and node (i + di, j + dj); 0 outside the grid
__device__ __forceinline__ double cf(const MgMat& A, int i, int j, int di, int dj) {
  const int mx = A.mx, my = A.my, idx = i * mx + j;
  if (di == 0 && dj == 0) return A.C[idx];
  if (di == 0) return dj > 0 ? (j + 1 < mx ? A.E[idx] : 0.0) : (j > 0 ? A.E[idx - 1] : 0.0);
  if (dj == 0) return di > 0 ? (i + 1 < my ? A.N[idx] : 0.0) : (i > 0 ? A.N[idx - mx] : 0.0);
  if (!A.nine) return 0.0;
  if (di > 0) {
    if (i + 1 >= my) return 0.0;
    return dj > 0 ? (j + 1 < mx ? A.NE[idx] : 0.0) : (j > 0 ? A.NW[idx] : 0.0);
  }
  if (i == 0) return 0.0;
  return dj > 0 ? (j + 1 < mx ? A.NW[idx - mx + 1] : 0.0) : (j > 0 ? A.NE[idx - mx - 1] : 0.0);
}

// sum over the neighbours of (i, j) of a_nb * X(nb), X given as a functor of the linear index
template <class X>
__device__ __forceinline__ double offsum(const MgMat& A, int i, int j, int idx, X x) {
  const int mx = A.mx, my = A.my;
  double s = 0.0;
  const bool w = j > 0, e = j + 1 < mx, so = i > 0, n = i + 1 < my;
  if (w) s = fma(A.E[idx - 1], x(idx - 1), s);
  if (e) s = fma(A.E[idx], x(idx + 1), s);
  if (so) s = fma(A.N[idx - mx], x(idx - mx), s);
  if (n) s = fma(A.N[idx], x(idx + mx), s);
  if (A.nine) {
    if (so && w) s = fma(A.NE[idx - mx - 1], x(idx - mx - 1), s);
    if (so && e) s = fma(A.NW[idx - mx + 1], x(idx - mx + 1), s);
    if (n && w) s = fma(A.NW[idx], x(idx + mx - 1), s);
    if (n && e) s = fma(A.NE[idx], x(idx + mx + 1), s);
  }
  return s;
}

// interpolation weight of fine node (i, j) towards coarse node (I, J) (coarse node = fine (2I+1, 2J+1)); 0 outside
__device__ __forceinline__ double pweight(const MgMat& A, int i, int j, int I, int J) {
  const int cy = A.my >> 1, cx = A.mx >> 1;
  if (I < 0 || I >= cy || J < 0 || J >= cx) return 0.0;
  const int di = i - (2 * I + 1), dj = j - (2 * J + 1);
  if (di < -1 || di > 1 || dj < -1 || dj > 1) return 0.0;
  if (di == 0 && dj == 0) return 1.0;
  const int idx = i * A.mx + j;
  int k;
  if (di == 0) k = dj > 0 ? 0 : 1;                 // node on a horizontal coarse line: weights (W, E)
  else if (dj == 0) k = di > 0 ? 0 : 1;            // node on a vertical coarse line: weights (S, N)
  else k = (di > 0 ? 0 : 2) + (dj > 0 ? 0 : 1);    // cell centre: weights (SW, SE, NW, NE)
  return A.pw[static_cast<size_t>(k) * A.n + idx];
}

// collapsed-stencil weights of a node on a horizontal / vertical coarse line (Dendy)
__device__ __forceinline__ void w_h(const MgMat& A, int i, int j, double& wW, double& wE) {
  const double ch = cf(A, i, j, 0, 0) + cf(A, i, j, 1, 0) + cf(A, i, j, -1, 0);
  wW = -(cf(A, i, j, 0, -1) + cf(A, i, j, 1, -1) + cf(A, i, j, -1, -1)) / ch;
  wE = -(cf(A, i, j, 0, 1) + cf(A, i, j, 1, 1) + cf(A, i, j, -1, 1)) / ch;
}
__device__ __forceinline__ void w_v(const MgMat& A, int i, int j, double& wS, double& wN) {
  const double cv = cf(A, i, j, 0, 0) + cf(A, i, j, 0, 1) + cf(A, i, j, 0, -1);
  wS = -(cf(A, i, j, -1, 0) + cf(A, i, j, -1, 1) + cf(A, i, j, -1, -1)) / cv;
  wN = -(cf(A, i, j, 1, 0) + cf(A, i, j, 1, 1) + cf(A, i, j, 1, -1)) / cv;
}

// ---------------------------------------------------------------------------------------------- setup kernels
// level 0 from the assembled CSR values: centre / east / north of every interior node; checks the hypotenuse entries
__global__ void k_mg_extract(const dfe::MeshDev M, const double* __restrict__ vals, int gx, MgMat A, int* flag) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= A.n) return;
  const int i = idx / A.mx, j = idx - i * A.mx;
  const int p = (i + 1) * (gx + 1) + (j + 1);
  double c = 0.0, e = 0.0, nn = 0.0;
  bool bad = false;
  for (int k = M.rowptr[p]; k < M.rowptr[p + 1]; ++k) {
    const int q = M.col[k];
    const double v = vals[k];
    if (q == p) c = v;
    else if (q == p + 1) e = v;
    else if (q == p + gx + 1) nn = v;
    else if (q == p - 1 || q == p - gx - 1) {}
    else if (v != 0.0) bad = true;            // hypotenuse neighbours p - gx, p + gx (or anything else): must be exact zeros
  }
  if (!(c > 0.0) || !isfinite(c)) bad = true;
  A.C[idx] = c;
  A.dinv[idx] = 1.0 / c;
  A.E[idx] = (j + 1 < A.mx) ? e : 0.0;        // couplings to Dirichlet nodes are not part of K_free
  A.N[idx] = (i + 1 < A.my) ? nn : 0.0;
  if (bad) *flag = 1;
}

__global__ void k_mg_weights(MgMat A) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= A.n) return;
  const int i = idx / A.mx, j = idx - i * A.mx;
  const size_t n = A.n;
  double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0;
  const bool oi = i & 1, oj = j & 1;
  if (oi && !oj) {
    w_h(A, i, j, w0, w1);
  } else if (!oi && oj) {
    w_v(A, i, j, w0, w1);
  } else if (!oi && !oj) {
    const double aW = cf(A, i, j, 0, -1), aE = cf(A, i, j, 0, 1), aS = cf(A, i, j, -1, 0), aN = cf(A, i, j, 1, 0);
    double wSW = 0, wNW = 0, wSE = 0, wNE = 0, sW = 0, sE = 0, nW = 0, nE = 0;
    if (j > 0) w_v(A, i, j - 1, wSW, wNW);          // west neighbour: (S, N) weights
    if (j + 1 < A.mx) w_v(A, i, j + 1, wSE, wNE);    // east neighbour
    if (i > 0) w_h(A, i - 1, j, sW, sE);            // south neighbour: (W, E) weights
    if (i + 1 < A.my) w_h(A, i + 1, j, nW, nE);      // north neighbour
    const double c = cf(A, i, j, 0, 0);
    w0 = -(cf(A, i, j, -1, -1) + aW * wSW + aS * sW) / c;   // SW
    w1 = -(cf(A, i, j, -1, 1) + aE * wSE + aS * sE) / c;    // SE
    w2 = -(cf(A, i, j, 1, -1) + aW * wNW + aN * nW) / c;    // NW
    w3 = -(cf(A, i, j, 1, 1) + aE * wNE + aN * nE) / c;     // NE
  }
  A.pw[idx] = w0;
  A.pw[n + idx] = w1;
  A.pw[2 * n + idx] = w2;
  A.pw[3 * n + idx] = w3;
}

// Galerkin coarse operator Ac = P^T A P in stencil form, one thread per coarse node
__global__ void k_mg_rap(MgMat A, MgMat Ac) {
  const int cidx = blockIdx.x * blockDim.x + threadIdx.x;
  if (cidx >= Ac.n) return;
  const int I = cidx / Ac.mx, J = cidx - I * Ac.mx;
  const int fi = 2 * I + 1, fj = 2 * J + 1;
  double acc[5] = {0, 0, 0, 0, 0};   // (0,0) (0,1) (1,0) (1,1) (1,-1)
  const int dI[5] = {0, 0, 1, 1, 1}, dJ[5] = {0, 1, 0, 1, -1};
  for (int pi = fi - 1; pi <= fi + 1; ++pi) {
    if (pi < 0 || pi >= A.my) continue;
    for (int pj = fj - 1; pj <= fj + 1; ++pj) {
      if (pj < 0 || pj >= A.mx) continue;
      const double wp = pweight(A, pi, pj, I, J);
      if (wp == 0.0) continue;
      for (int di = -1; di <= 1; ++di) {
        const int qi = pi + di;
        if (qi < 0 || qi >= A.my) continue;
        for (int dj = -1; dj <= 1; ++dj) {
          const int qj = pj + dj;
          if (qj < 0 || qj >= A.mx) continue;
          if (!A.nine && di != 0 && dj != 0) continue;
          const double a = cf(A, pi, pj, di, dj);
          if (a == 0.0) continue;
          const double wa = wp * a;
#pragma unroll
          for (int d = 0; d < 5; ++d) acc[d] = fma(wa, pweight(A, qi, qj, I + dI[d], J + dJ[d]), acc[d]);
        }
      }
    }
  }
  Ac.C[cidx] = acc[0];
  Ac.dinv[cidx] = 1.0 / acc[0];
  Ac.E[cidx] = (J + 1 < Ac.mx) ? acc[1] : 0.0;
  Ac.N[cidx] = (I + 1 < Ac.my) ? acc[2] : 0.0;
  Ac.NE[cidx] = (I + 1 < Ac.my && J + 1 < Ac.mx) ? acc[3] : 0.0;
  Ac.NW[cidx] = (I + 1 < Ac.my && J > 0) ? acc[4] : 0.0;
}

// explicit inverse of the coarsest operator (<= 32 unknowns): Gauss-Jordan without pivoting (SPD), one thread
__global__ void k_mg_coarsest(MgMat A, double* cinv, int* flag) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  __shared__ double a[MG_COARSEST * MG_COARSEST];
  const int n = A.n;
  for (int r = 0; r < n; ++r) {
    const int i = r / A.mx, j = r - i * A.mx;
    for (int c = 0; c < n; ++c) {
      a[r * n + c] = 0.0;
      cinv[r * n + c] = r == c ? 1.0 : 0.0;
    }
    for (int di = -1; di <= 1; ++di)
      for (int dj = -1; dj <= 1; ++dj) {
        const int qi = i + di, qj = j + dj;
        if (qi < 0 || qi >= A.my || qj < 0 || qj >= A.mx) continue;
        a[r * n + qi * A.mx + qj] = cf(A, i, j, di, dj);
      }
  }
  for (int k = 0; k < n; ++k) {
    const double piv = a[k * n + k];
    if (!(piv > 0.0) || !isfinite(piv)) { *flag = 2; return; }
    const double ip = 1.0 / piv;
    for (int c = 0; c < n; ++c) { a[k * n + c] *= ip; cinv[k * n + c] *= ip; }
    for (int r = 0; r < n; ++r) {
      if (r == k) continue;
      const double f = a[r * n + k];
      if (f == 0.0) continue;
      for (int c = 0; c < n; ++c) {
        a[r * n + c] = fma(-f, a[k * n + c], a[r * n + c]);
        cinv[r * n + c] = fma(-f, cinv[k * n + c], cinv[r * n + c]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- solve kernel
struct MgArgs {
  MgHier H;
  MgVec v[MG_MAXL];
  const double* rhs;
  double *x, *p0, *p1, *q;
  double* out;          // [0] iterations, [1] relres, [2] status (0 ok, 4 not converged, 5 breakdown, 7 barrier timeout),
                        // [3] 1 if the breakdown is a non-finite rhs
  double* slots;
  int* abort_flag;
  double tol;
  long long maxit;
  int nu, backoff;
  double omega[8];      // damping of smoothing sweep 1 .. nu (Chebyshev weights, see mg_omegas)
};

// contiguous range of the n nodes of a level owned by this CTA
__device__ __forceinline__ void cta_range(int n, int& lo, int& hi) {
  const int G = gridDim.x;
  int chunk = (n + G - 1) / G;
  chunk = (chunk + 31) & ~31;
  lo = blockIdx.x * chunk;
  if (lo > n) lo = n;
  hi = lo + chunk < n ? lo + chunk : n;
}

// levels with at most TAIL_N unknowns are handled by CTA 0 alone, matrices and work vectors in its shared memory
constexpr int TAIL_N = 1024;

#define MG_KERNEL_NS mg768
#define MG_KERNEL_MT 768
#include "dfe_mg_kernel.cuh"
#undef MG_KERNEL_NS
#undef MG_KERNEL_MT
#define MG_KERNEL_NS mg512
#define MG_KERNEL_MT 512
#include "dfe_mg_kernel.cuh"
#undef MG_KERNEL_NS
#undef MG_KERNEL_MT
constexpr int MG_SMALL_N = 65536;   // grids up to this size run the 512-thread kernel

// ---------------------------------------------------------------------------------------------- host side
struct Dims {
  int L;
  int my[MG_MAXL], mx[MG_MAXL];
};

// level sizes of the interior grid of a gx x gy quad mesh; L = 0 if the hierarchy does not end on a small grid
Dims mg_dims(int gx, int gy) {
  Dims d{};
  int my = gy - 1, mx = gx - 1;
  if (my < 1 || mx < 1) return d;
  int L = 0;
  while (L < MG_MAXL) {
    d.my[L] = my;
    d.mx[L] = mx;
    ++L;
    if (static_cast<long long>(my) * mx <= MG_COARSEST) {
      d.L = L;
      return d;
    }
    if (my < 2 || mx < 2) break;   // cannot coarsen further, and the grid is still large (extreme aspect ratio)
    my >>= 1;
    mx >>= 1;
  }
  d.L = 0;
  return d;
}

inline size_t al(size_t bytes) { return (bytes + 255) / 256 * 256; }

// shared memory of the solve kernel: matrices and work vectors of the tail levels (must mirror k_mgpcg)
size_t tail_smem_bytes(const Dims& d) {
  int lc = d.L - 1;
  while (lc > 1 && static_cast<long long>(d.my[lc - 1]) * d.mx[lc - 1] <= TAIL_N) --lc;
  size_t dbl = 0;
  for (int l = lc; l < d.L; ++l) {
    const size_t n = static_cast<size_t>(d.my[l]) * d.mx[l];
    dbl += 6 * n + (l + 1 < d.L ? 4 * n : 0) + n + (l > lc ? 3 * n : 0);
  }
  return dbl * sizeof(double) + 64;
}

// carve the hierarchy buffer; returns the total size.  base may be null (size query).
size_t carve_hier(const Dims& d, unsigned char* base, MgHier* H) {
  size_t off = 0;
  auto take = [&](size_t n_doubles) {
    double* p = base ? reinterpret_cast<double*>(base + off) : nullptr;
    off += al(n_doubles * sizeof(double));
    return p;
  };
  if (H) { H->L = d.L; H->nc = d.my[d.L - 1] * d.mx[d.L - 1]; }
  for (int l = 0; l < d.L; ++l) {
    const size_t n = static_cast<size_t>(d.my[l]) * d.mx[l];
    MgMat M{};
    M.my = d.my[l]; M.mx = d.mx[l]; M.n = static_cast<int>(n); M.nine = l > 0;
    M.C = take(n); M.dinv = take(n); M.E = take(n); M.N = take(n);
    if (l > 0) { M.NE = take(n); M.NW = take(n); }
    if (l + 1 < d.L) M.pw = take(4 * n);
    if (H) H->lev[l] = M;
  }
  double* cinv = take(static_cast<size_t>(MG_COARSEST) * MG_COARSEST);
  int* flag = base ? reinterpret_cast<int*>(base + off) : nullptr;
  off += 256;
  if (H) { H->cinv = cinv; H->flag = flag; }
  return off;
}

struct MgWs {
  size_t vec[MG_MAXL][4], x_unused, p0, p1, q, slots, out, abort_flag, total;
};
void plan_ws(const Dims& d, MgWs* w) {
  size_t off = 0;
  for (int l = 0; l < d.L; ++l) {
    const size_t n = static_cast<size_t>(d.my[l]) * d.mx[l];
    for (int k = 0; k < 4; ++k) { w->vec[l][k] = off; off += al(n * sizeof(double)); }
  }
  const size_t n0 = static_cast<size_t>(d.my[0]) * d.mx[0];
  w->p0 = off; off += al(n0 * sizeof(double));
  w->p1 = off; off += al(n0 * sizeof(double));
  w->q = off; off += al(n0 * sizeof(double));
  w->slots = off; off += al(6 * 148 * 8 * sizeof(double));
  w->out = off; off += 256;
  w->abort_flag = off; off += 256;
  w->total = off;
}

int mg_enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (m->grid_nx <= 0 || mg_dims(m->grid_nx, m->grid_ny).L < 2) {
    dfe::set_error("%s: the mesh does not have the structure of FEMesh.rectangle() with Dirichlet sides (dfe_mg_supported == 0)", who);
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}

inline unsigned nblk(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

}  // namespace

extern "C" int dfe_mg_supported(const dfe_mesh* m) {
  if (!m || m->grid_nx <= 0) return 0;
  const Dims d = mg_dims(m->grid_nx, m->grid_ny);
  return (d.L >= 2 && static_cast<long long>(d.my[0]) * d.mx[0] >= 1024) ? 1 : 0;
}

extern "C" size_t dfe_mg_hierarchy_bytes(const dfe_mesh* m) {
  if (!m || m->grid_nx <= 0) return 0;
  const Dims d = mg_dims(m->grid_nx, m->grid_ny);
  if (d.L < 2) return 0;
  return carve_hier(d, nullptr, nullptr);
}

extern "C" size_t dfe_mg_workspace_bytes(const dfe_mesh* m) {
  if (!m || m->grid_nx <= 0) return 0;
  const Dims d = mg_dims(m->grid_nx, m->grid_ny);
  if (d.L < 2) return 0;
  MgWs w;
  plan_ws(d, &w);
  return w.total;
}

extern "C" int dfe_mg_setup(const dfe_mesh* m, const double* vals_full, void* hier, size_t hier_bytes, void* stream) {
  int prev;
  int rc = mg_enter(m, "dfe_mg_setup", &prev);
  if (rc) return rc;
  const Dims d = mg_dims(m->grid_nx, m->grid_ny);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  MgHier H{};
  if (!vals_full || !hier) {
    dfe::set_error("dfe_mg_setup: null argument");
    rc = DFE_ERR_INVALID;
  } else if (hier_bytes < carve_hier(d, static_cast<unsigned char*>(hier), &H)) {
    dfe::set_error("dfe_mg_setup: hierarchy buffer %zu bytes < required %zu", hier_bytes, carve_hier(d, nullptr, nullptr));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaError_t e = cudaMemsetAsync(H.flag, 0, sizeof(int), st);
    if (e == cudaSuccess) {
      k_mg_extract<<<nblk(H.lev[0].n, 256), 256, 0, st>>>(m->dev, vals_full, m->grid_nx, H.lev[0], H.flag);
      for (int l = 0; l + 1 < H.L; ++l) {
        k_mg_weights<<<nblk(H.lev[l].n, 256), 256, 0, st>>>(H.lev[l]);
        k_mg_rap<<<nblk(H.lev[l + 1].n, 128), 128, 0, st>>>(H.lev[l], H.lev[l + 1]);
      }
      k_mg_coarsest<<<1, 32, 0, st>>>(H.lev[H.L - 1], H.cinv, H.flag);
      e = cudaGetLastError();
    }
    int flag = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&flag, H.flag, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      dfe::set_error("dfe_mg_setup: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    } else if (flag == 1) {
      dfe::set_error("dfe_mg_setup: K_free is not numerically a 5-point operator on the node grid (distorted coordinates or a "
                     "non-positive diagonal): use dfe_pcg");
      rc = DFE_ERR_UNSUPPORTED;
    } else if (flag == 2) {
      dfe::set_error("dfe_mg_setup: the coarsest Galerkin operator is not positive definite: use dfe_pcg");
      rc = DFE_ERR_UNSUPPORTED;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_mg_pcg(const dfe_mesh* m, const void* hier, const double* rhs, double* x, double tol, int64_t maxit,
                          int nu, int64_t* iters_host, double* relres_host, void* ws, size_t ws_bytes, void* stream) {
  int prev;
  int rc = mg_enter(m, "dfe_mg_pcg", &prev);
  if (rc) return rc;
  if (iters_host) *iters_host = 0;
  if (relres_host) *relres_host = 0.0;
  const Dims d = mg_dims(m->grid_nx, m->grid_ny);
  MgWs w;
  plan_ws(d, &w);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!hier || !rhs || !x || !ws || !(tol > 0.0) || maxit < 1 || nu < 1 || nu > 4) {
    dfe::set_error("dfe_mg_pcg: bad argument (null pointer, tol <= 0, maxit < 1 or nu outside 1..4)");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < w.total) {
    dfe::set_error("dfe_mg_pcg: workspace %zu bytes < required %zu", ws_bytes, w.total);
    rc = DFE_ERR_WORKSPACE;
  } else {
    MgArgs* Ap = new MgArgs();   // ~1.5 KB of kernel parameters
    MgArgs& R = *Ap;
    carve_hier(d, const_cast<unsigned char*>(static_cast<const unsigned char*>(hier)), &R.H);
    unsigned char* b = static_cast<unsigned char*>(ws);
    for (int l = 0; l < d.L; ++l) {
      R.v[l].b = reinterpret_cast<double*>(b + w.vec[l][0]);
      R.v[l].r = reinterpret_cast<double*>(b + w.vec[l][1]);
      R.v[l].xa = reinterpret_cast<double*>(b + w.vec[l][2]);
      R.v[l].xb = reinterpret_cast<double*>(b + w.vec[l][3]);
    }
    R.rhs = rhs;
    R.x = x;
    R.p0 = reinterpret_cast<double*>(b + w.p0);
    R.p1 = reinterpret_cast<double*>(b + w.p1);
    R.q = reinterpret_cast<double*>(b + w.q);
    R.slots = reinterpret_cast<double*>(b + w.slots);
    R.out = reinterpret_cast<double*>(b + w.out);
    R.abort_flag = reinterpret_cast<int*>(b + w.abort_flag);
    R.tol = tol;
    R.maxit = maxit;
    R.nu = nu;
    mg_omegas(nu, R.omega);
    static const int backoff = [] { const char* e = getenv("DFE_PCG_BACKOFF"); return e ? atoi(e) : 250; }();
    R.backoff = backoff;
    int per_sm = 0;
    const size_t smem = tail_smem_bytes(d);
    // CTA size: 512 threads for small grids (latency-bound: fewer, fatter threads), 768 otherwise; DFE_MG_MT=768 / 512 forces one
    const char* mte = getenv("DFE_MG_MT");
    const bool small = mte ? atoi(mte) == 512 : R.H.lev[0].n <= MG_SMALL_N;
    void* const kern = small ? reinterpret_cast<void*>(mg512::k_mgpcg) : reinterpret_cast<void*>(mg768::k_mgpcg);
    const int MT = small ? mg512::MT : mg768::MT;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, MT, smem);
    long long grid = static_cast<long long>(per_sm > 0 ? 1 : 0) * m->sm_count;   // one CTA per SM
    const long long want = (static_cast<long long>(R.H.lev[0].n) + MT - 1) / MT;
    if (grid > want) grid = want;
    if (grid > 148 * 8) grid = 148 * 8;
    if (e == cudaSuccess && grid < 1) {
      dfe::set_error("dfe_mg_pcg: kernel does not fit on the device");
      rc = DFE_ERR_CUDA;
    }
    if (rc == DFE_OK) {
      if (e == cudaSuccess) e = cudaMemsetAsync(R.slots, 0xFF, 6 * static_cast<size_t>(grid) * sizeof(double), st);
      if (e == cudaSuccess) e = cudaMemsetAsync(R.abort_flag, 0, sizeof(int), st);
      void* args[] = {&R};
      if (e == cudaSuccess)
        e = cudaLaunchCooperativeKernel(kern, dim3(static_cast<unsigned>(grid)), dim3(MT), args, smem, st);
      double out[4] = {0, 0, 0, 0};
      if (e == cudaSuccess) e = cudaMemcpyAsync(out, R.out, sizeof out, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) {
        dfe::set_error("dfe_mg_pcg: %s", cudaGetErrorString(e));
        rc = DFE_ERR_CUDA;
      } else {
        if (iters_host) *iters_host = static_cast<int64_t>(out[0]);
        if (relres_host) *relres_host = out[1];
        if (out[2] == 4.0) {
          dfe::set_error("dfe_mg_pcg: not converged after %lld iterations (relative residual %.3e, tol %.3e)",
                         static_cast<long long>(out[0]), out[1], tol);
          rc = DFE_ERR_NOT_CONVERGED;
        } else if (out[2] == 5.0 && out[3] != 0.0) {
          dfe::set_error("dfe_mg_pcg: breakdown at iteration 0: the right-hand side has a non-finite entry (inf or NaN)");
          rc = DFE_ERR_BREAKDOWN;
        } else if (out[2] == 5.0) {
          dfe::set_error("dfe_mg_pcg: breakdown at iteration %lld (r^T M r <= 0, p^T K p <= 0 or non-finite)",
                         static_cast<long long>(out[0]));
          rc = DFE_ERR_BREAKDOWN;
        } else if (out[2] == 7.0) {
          dfe::set_error("dfe_mg_pcg: a grid barrier waited longer than its bound (lost co-resident CTA?)");
          rc = DFE_ERR_CUDA;
        }
      }
    }
    delete Ap;
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}
