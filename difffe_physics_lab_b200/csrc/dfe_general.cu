// General (CSR) path: P1 assembly, Dirichlet elimination, scatter/gather and the element-gradient
// kernels for 2-D triangle meshes and for 1-D meshes that are not chains.
//
//   k_assemble   diffhe/solver.py:82-96 (1-D) and :112-145 (2-D): one thread per matrix row walks
//                the elements around its node in ascending element id — the reference's own
//                accumulation order — so K (structural CSR) and F are bit-identical to the dense
//                reference without float atomics.  All arithmetic uses explicit round-to-nearest
//                intrinsics in the reference's operation order (no FMA contraction).
//   k_eliminate  solver.py:162-171: F_free = F[free] - sum_d K[free,d] g_d in dict order,
//                1/diag(K_free), CSR values of K_free;  k_fill_sell copies K_free into SELL-32.
//   k_scatter / k_gather   solver.py:177-181 and the restriction of gbar to free rows.
//   k_grad_elem / k_grad_f the closed-form backward of the assembly (SURVEY §8a row A8).
#include <cstdint>
#include <cstdlib>

#include "dfe_internal.h"

namespace {

using dfe::MeshDev;
#include "dfe_assemble_row.cuh"   // AREA_EPS, elem2d, p2_tri_of, assemble_row (P2: dfe_p2.cuh)

__global__ void k_assemble(const MeshDev M, const double* __restrict__ kappa, int per_elem,
                           const double* __restrict__ f, double* __restrict__ vals, double* __restrict__ F) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_nodes) return;
  if (M.rowptr[p + 1] - M.rowptr[p] <= ROWMAX) assemble_row<true>(M, p, kappa, per_elem, f, vals, F);
  else assemble_row<false>(M, p, kappa, per_elem, f, vals, F);
}

// ---- structured variant for meshes with the element pattern of FEMesh.rectangle(gx, gy) (mesh.py:92-120).
// The adjacency of a node is known in closed form there: node p = (r, c) touches, in ascending element id,
//   quad (r-1, c-1) tri 1 = [S, C, W]      quad (r-1, c) tri 0 = [S, SE, C]   and tri 1 = [SE, E, C]
//   quad (r, c-1)   tri 0 = [W, C, NW]     and tri 1 = [C, N, NW]             quad (r, c) tri 0 = [C, E, N]
// (S = p-gx-1, SE = p-gx, W = p-1, E = p+1, NW = p+gx, N = p+gx+1 — which is also the ascending column order of the
// CSR row), so the kernel needs no adjacency lists, no slot tables and no connectivity: it reads coordinates, kappa
// and f (coalesced along a mesh line, neighbours from L1), accumulates the row in registers in the reference's
// element order with the reference's operation order, and writes the row once — through shared memory, so that the
// stores of a CTA are one contiguous coalesced stream.  Same bits as k_assemble (and as the reference's dense K, F).
constexpr int AG_T = 256;

#include "dfe_exact.cuh"   // div_markstein, mid_range, div3

__device__ __forceinline__ void tri_row(const double (&x)[3], const double (&y)[3], int loc, double kap, double (&k)[3],
                                        double& area, bool& keep) {
  const double t1 = __dmul_rn(__dsub_rn(x[1], x[0]), __dsub_rn(y[2], y[0]));
  const double t2 = __dmul_rn(__dsub_rn(x[2], x[0]), __dsub_rn(y[1], y[0]));
  area = __dmul_rn(0.5, fabs(__dsub_rn(t1, t2)));          // solver.py:119
  keep = !(area < AREA_EPS);                                // :120-121
  const double b[3] = {__dsub_rn(y[1], y[2]), __dsub_rn(y[2], y[0]), __dsub_rn(y[0], y[1])};
  const double c[3] = {__dsub_rn(x[2], x[1]), __dsub_rn(x[0], x[2]), __dsub_rn(x[1], x[0])};
  const double den = __dmul_rn(4.0, area);
  const bool fast = mid_range(den);
  const double rden = fast ? __drcp_rn(den) : 0.0;
#pragma unroll
  for (int q = 0; q < 3; ++q) {   // k_pq = kappa*(b_p b_q + c_p c_q)/(4 area)   (:139)
    const double num = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[loc], b[q]), __dmul_rn(c[loc], c[q])));
    k[q] = (fast && (num == 0.0 || mid_range(num))) ? div_markstein(num, den, rden) : __ddiv_rn(num, den);
  }
}

__global__ void __launch_bounds__(AG_T, 3) k_assemble_grid(const MeshDev M, int gx, int gy, const double* __restrict__ kappa,
                                                        int per_elem, const double* __restrict__ f,
                                                        double* __restrict__ vals, double* __restrict__ F) {
  __shared__ double stage[7 * AG_T];
  const int p0 = blockIdx.x * AG_T;
  const int p = p0 + threadIdx.x;
  const int np1 = gx + 1;
  const bool live = p < M.n_nodes;
  const int pend = min(p0 + AG_T, M.n_nodes);
  const int base0 = M.rowptr[p0], base1 = M.rowptr[pend];
  if (live) {
    const int r = p / np1, cc = p - r * np1;
    const bool hasS = r > 0, hasN = r < gy, hasW = cc > 0, hasE = cc < gx;
    // slots: 0 S, 1 SE, 2 W, 3 C, 4 E, 5 NW, 6 N
    const int nid[7] = {p - np1, p - gx, p - 1, p, p + 1, p + gx, p + np1};
    const bool ex[7] = {hasS, hasS && hasE, hasW, true, hasE, hasN && hasW, hasN};
    // (the kernel is bound by the latency of its dependent FP64 chains, ncu: FP64 pipe 37 %, 25 % occupancy at 96
    // registers — f is therefore re-read per element from L1 instead of being held, and the register bound allows three CTAs per SM)
    double xs[7], ys[7], v[7];
    const double2* xy = reinterpret_cast<const double2*>(M.nodes);
#pragma unroll
    for (int s = 0; s < 7; ++s) {
      v[s] = 0.0;
      xs[s] = ys[s] = 0.0;
      if (ex[s]) {
        const double2 c2 = xy[nid[s]];
        xs[s] = c2.x;
        ys[s] = c2.y;
      }
    }
    double Fp = 0.0;
    // (element exists, element id, node slots in element order, position of p)
    const int qS = (r - 1) * gx + cc, qN = r * gx + cc;   // quads (r-1, c) and (r, c)
    const bool eex[6] = {hasS && hasW, hasS && hasE, hasS && hasE, hasN && hasW, hasN && hasW, hasN && hasE};
    const int eid[6] = {2 * (qS - 1) + 1, 2 * qS, 2 * qS + 1, 2 * (qN - 1), 2 * (qN - 1) + 1, 2 * qN};
    const int en[6][3] = {{0, 3, 2}, {0, 1, 3}, {1, 4, 3}, {2, 3, 5}, {3, 6, 5}, {3, 4, 6}};
    const int eloc[6] = {1, 2, 2, 1, 0, 0};
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      if (!eex[t]) continue;
      const double kap = kappa[per_elem ? eid[t] : 0];
      const double ex3[3] = {xs[en[t][0]], xs[en[t][1]], xs[en[t][2]]};
      const double ey3[3] = {ys[en[t][0]], ys[en[t][1]], ys[en[t][2]]};
      double k[3], area;
      bool keep;
      tri_row(ex3, ey3, eloc[t], kap, k, area, keep);
      if (!keep) continue;
#pragma unroll
      for (int q = 0; q < 3; ++q) v[en[t][q]] = __dadd_rn(v[en[t][q]], k[q]);
      // F_p += area/3 * (f_i+f_j+f_k)/3   (:143-145)
      const double fc = div3(__dadd_rn(__dadd_rn(f[nid[en[t][0]]], f[nid[en[t][1]]]), f[nid[en[t][2]]]));
      Fp = __dadd_rn(Fp, __dmul_rn(div3(area), fc));
    }
    F[p] = Fp;
    int k = M.rowptr[p] - base0;
#pragma unroll
    for (int s = 0; s < 7; ++s)
      if (ex[s]) stage[k++] = v[s];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < base1 - base0; i += AG_T) vals[base0 + i] = stage[i];
}

// ---- element-parallel structured assembly (default on rectangle() patterns).
// k_assemble_grid above computes every triangle three times (once per vertex row) and every row needs 18 divisions:
// ncu showed it FP64-latency bound (FP64 pipe 35 %, 24 % occupancy, 86 us for the 134 MB of config 4).  Here a CTA owns a
// tile of AQ_R x AQ_C QUADS and the (AQ_R - 1) x (AQ_C - 1) nodes whose six triangles all lie in the tile (tiles overlap
// by one quad row / column: 18 % redundant element work instead of 200 %).  Phase 1: one thread per quad computes the two
// element matrices ONCE — six entries each (the reference's K is bitwise symmetric: b_p b_q + c_p c_q commutes), one
// reciprocal and Markstein-corrected quotients — plus the load term, into shared memory.  Phase 2: one thread per node
// adds the entries of its row in ascending element order (the reference's accumulation order), stages the row, and
// the CTA writes its CSR values as contiguous streams.  Same bits as k_assemble (tests: bit-exact vs the dense reference).
constexpr int AQ_R = 8, AQ_C = 32, AQ_T = AQ_R * AQ_C;       // quads per tile = threads
constexpr int AN_R = AQ_R - 1, AN_C = AQ_C - 1, AN_T = AN_R * AN_C;   // nodes per tile

// is v exactly zero, or safely inside the range where the Markstein residuals neither overflow nor underflow?
__device__ __forceinline__ bool zero_or_mid(double v) {
  const unsigned hi = static_cast<unsigned>(__double2hiint(v)) & 0x7fffffffu;
  const unsigned e = hi >> 20;
  return (e - 558u) <= 930u || (hi | static_cast<unsigned>(__double2loint(v))) == 0u;   // 2^-465 .. 2^465, or +-0
}
// a / b from y = RN(1/b), correctly rounded (see dfe_exact.cuh); a zero numerator may lose its sign, which no
// accumulation that starts from +0 can observe
__device__ __forceinline__ double div_m(double a, double b, double y) {
  const double q0 = __dmul_rn(a, y);
  const double q1 = fma(fma(-b, q0, a), y, q0);
  return fma(fma(-b, q1, a), y, q1);
}

// kappa is exactly zero or in [2^-170, 2^170] (with dfe_mesh::topo_geo_mid: every numerator then is 0 or in [2^-463, 2^411])
__device__ __forceinline__ bool kappa_zero_or_mid(double v) {
  const unsigned hi = static_cast<unsigned>(__double2hiint(v)) & 0x7fffffffu;
  return ((hi >> 20) - 853u) <= 340u || (hi | static_cast<unsigned>(__double2loint(v))) == 0u;
}

// element matrix (k00 k01 k02 k11 k12 k22) and load term (area/3) * (f_i + f_j + f_k)/3 of one triangle, solver.py:119-145.
// GEO: the handle has verified the range of the geometry once (dfe_mesh::topo_geo_mid), so only kappa and the load sum are
// range-checked per call; otherwise every numerator is.
template <bool GEO>
__device__ __forceinline__ void tri_full(const double (&x)[3], const double (&y)[3], double kap, const double (&fv)[3],
                                         double (&k)[6], double& fterm) {
  const double b[3] = {__dsub_rn(y[1], y[2]), __dsub_rn(y[2], y[0]), __dsub_rn(y[0], y[1])};
  const double c[3] = {__dsub_rn(x[2], x[1]), __dsub_rn(x[0], x[2]), __dsub_rn(x[1], x[0])};
  // :119  (x_j - x_i)(y_k - y_i) - (x_k - x_i)(y_j - y_i) = c2 b1 - (-c1)(-b2): negation is exact, the products are the same bits
  const double t1 = __dmul_rn(c[2], b[1]);
  const double t2 = __dmul_rn(c[1], b[2]);
  const double area = __dmul_rn(0.5, fabs(__dsub_rn(t1, t2)));
  const double den = __dmul_rn(4.0, area);
  double num[6];
  num[0] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[0], b[0]), __dmul_rn(c[0], c[0])));   // :139
  num[1] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[0], b[1]), __dmul_rn(c[0], c[1])));
  num[2] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[0], b[2]), __dmul_rn(c[0], c[2])));
  num[3] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[1], b[1]), __dmul_rn(c[1], c[1])));
  num[4] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[1], b[2]), __dmul_rn(c[1], c[2])));
  num[5] = __dmul_rn(kap, __dadd_rn(__dmul_rn(b[2], b[2]), __dmul_rn(c[2], c[2])));
  const double fsum = __dadd_rn(__dadd_rn(fv[0], fv[1]), fv[2]);
  bool ok;
  if (GEO) {
    ok = kappa_zero_or_mid(kap) && zero_or_mid(fsum);
  } else {
    ok = zero_or_mid(den) && den != 0.0 && zero_or_mid(fsum) && zero_or_mid(area);
#pragma unroll
    for (int i = 0; i < 6; ++i) ok = ok && zero_or_mid(num[i]);
  }
  if (area < AREA_EPS) {                                          // :120-121 — contributes nothing (adds +0)
#pragma unroll
    for (int i = 0; i < 6; ++i) k[i] = 0.0;
    fterm = 0.0;
  } else if (ok) {
    const double rden = __drcp_rn(den);
    constexpr double third = 0.333333333333333314829616256247;   // RN(1/3)
#pragma unroll
    for (int i = 0; i < 6; ++i) k[i] = div_m(num[i], den, rden);
    fterm = __dmul_rn(div_m(area, 3.0, third), div_m(fsum, 3.0, third));   // :143-145
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) k[i] = __ddiv_rn(num[i], den);
    fterm = __dmul_rn(__ddiv_rn(area, 3.0), __ddiv_rn(fsum, 3.0));
  }
}

template <bool GEO>
__global__ void __launch_bounds__(AQ_T, 4) k_assemble_tile(const MeshDev M, int gx, int gy, const double* __restrict__ kappa,
                                                        int per_elem, const double* __restrict__ f,
                                                        double* __restrict__ vals, double* __restrict__ F) {
  __shared__ double tri[2][7][AQ_T];          // [triangle of the quad][k00 k01 k02 k11 k12 k22 fterm][quad]
  __shared__ double stage[AN_R][AN_C * 7];    // CSR values of one node-row segment, compact
  __shared__ int segbase[AN_R], seglen[AN_R];
  const int tid = threadIdx.x;
  const int np1 = gx + 1;
  const int R0 = blockIdx.y * AN_R, C0 = blockIdx.x * AN_C;   // first node of the tile
  // ---------------- phase 1: quad (R0 - 1 + qr, C0 - 1 + qc)
  {
    const int qr = tid / AQ_C, qc = tid % AQ_C;
    const int gr = R0 - 1 + qr, gc = C0 - 1 + qc;
    if (gr >= 0 && gr < gy && gc >= 0 && gc < gx) {
      const int a = gr * np1 + gc;            // corners a, b = a + 1, c = a + gx + 2, d = a + gx + 1  (mesh.py:105-113)
      const double2* xy = reinterpret_cast<const double2*>(M.nodes);
      const double2 pa = xy[a], pb = xy[a + 1], pc = xy[a + np1 + 1], pd = xy[a + np1];
      const double fa = f[a], fb = f[a + 1], fc = f[a + np1 + 1], fd = f[a + np1];
      const int e0 = 2 * (gr * gx + gc);
      double k0 = kappa[0], k1 = k0;
      if (per_elem) {
        const double2 kk = *reinterpret_cast<const double2*>(kappa + e0);
        k0 = kk.x;
        k1 = kk.y;
      }
      double k[6], ft;
      {   // triangle 0 = [a, b, d]
        const double x[3] = {pa.x, pb.x, pd.x}, y[3] = {pa.y, pb.y, pd.y}, fv[3] = {fa, fb, fd};
        tri_full<GEO>(x, y, k0, fv, k, ft);
#pragma unroll
        for (int i = 0; i < 6; ++i) tri[0][i][tid] = k[i];
        tri[0][6][tid] = ft;
      }
      {   // triangle 1 = [b, c, d]
        const double x[3] = {pb.x, pc.x, pd.x}, y[3] = {pb.y, pc.y, pd.y}, fv[3] = {fb, fc, fd};
        tri_full<GEO>(x, y, k1, fv, k, ft);
#pragma unroll
        for (int i = 0; i < 6; ++i) tri[1][i][tid] = k[i];
        tri[1][6][tid] = ft;
      }
    }
  }
  // ---------------- phase 2: node (R0 + nr, C0 + nc)
  const int nr = tid / AN_C, nc = tid - nr * AN_C;
  const int r = R0 + nr, cc = C0 + nc;
  const bool live = tid < AN_T && r <= gy && cc <= gx;
  const int p = r * np1 + cc;
  int rp = 0;
  if (live) rp = M.rowptr[p];
  if (tid < AN_T && nc == 0) {
    const bool rowlive = r <= gy && C0 <= gx;
    const int last = min(C0 + AN_C, np1);   // one past the last node of the segment
    segbase[nr] = rowlive ? rp : 0;
    seglen[nr] = rowlive ? M.rowptr[r * np1 + last] - rp : 0;
  }
  __syncthreads();
  if (live) {
    const bool hasS = r > 0, hasN = r < gy, hasW = cc > 0, hasE = cc < gx;
    // row slots: 0 S, 1 SE, 2 W, 3 C, 4 E, 5 NW, 6 N (ascending column order of the CSR row)
    const bool ex[7] = {hasS, hasS && hasE, hasW, true, hasE, hasN && hasW, hasN};
    double v[7];
#pragma unroll
    for (int s = 0; s < 7; ++s) v[s] = 0.0;
    double Fp = 0.0;
    // adjacent triangles in ascending element id: (quad in the tile, triangle, slots of its three nodes, row of p)
    const int qSW = nr * AQ_C + nc, qSE = qSW + 1, qNW = qSW + AQ_C, qNE = qNW + 1;
    const bool eex[6] = {hasS && hasW, hasS && hasE, hasS && hasE, hasN && hasW, hasN && hasW, hasN && hasE};
    const int eq[6] = {qSW, qSE, qSE, qNW, qNW, qNE};
    const int et[6] = {1, 0, 1, 0, 1, 0};
    const int en[6][3] = {{0, 3, 2}, {0, 1, 3}, {1, 4, 3}, {2, 3, 5}, {3, 6, 5}, {3, 4, 6}};
    const int eloc[6] = {1, 2, 2, 1, 0, 0};
    const int sym[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      if (!eex[t]) continue;
#pragma unroll
      for (int q = 0; q < 3; ++q) v[en[t][q]] = __dadd_rn(v[en[t][q]], tri[et[t]][sym[eloc[t]][q]][eq[t]]);
      Fp = __dadd_rn(Fp, tri[et[t]][6][eq[t]]);
    }
    F[p] = Fp;
    int k = rp - segbase[nr];
#pragma unroll
    for (int s = 0; s < 7; ++s)
      if (ex[s]) stage[nr][k++] = v[s];
  }
  __syncthreads();
#pragma unroll
  for (int sr = 0; sr < AN_R; ++sr) {
    const int len = seglen[sr];
    if (tid < len) vals[segbase[sr] + tid] = stage[sr][tid];
  }
}

__global__ void k_eliminate(const MeshDev M, const double* __restrict__ vals, const double* __restrict__ F,
                            double* __restrict__ vals_free, double* __restrict__ F_free,
                            double* __restrict__ dinv) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= M.n_free) return;
  double Fr = F[M.free_nodes[r]];
  for (int t = M.lift_ptr[r]; t < M.lift_ptr[r + 1]; ++t)
    Fr = __dsub_rn(Fr, __dmul_rn(vals[M.lift_src[t]], M.lift_g[t]));  // solver.py:169
  F_free[r] = Fr;
  const int ds = M.diag_src[r];
  dinv[r] = 1.0 / (ds >= 0 ? vals[ds] : 0.0);
  if (vals_free)
    for (int k = M.rowptr_f[r]; k < M.rowptr_f[r + 1]; ++k) vals_free[k] = vals[M.src_f[k]];
}

__global__ void k_fill_sell(const MeshDev M, const double* __restrict__ vals, double* __restrict__ sell_vals) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < M.sell_nnz; i += gridDim.x * blockDim.x) {
    const int s = M.sell_src[i];
    sell_vals[i] = s >= 0 ? vals[s] : 0.0;
  }
}

__global__ void k_scatter(const MeshDev M, const double* __restrict__ x, int zero_bc, double* __restrict__ u) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M.n_free) u[M.free_nodes[i]] = x[i];
  if (i < M.n_dir) u[M.dir_idx[i]] = zero_bc ? 0.0 : M.dir_val[i];
}

__global__ void k_gather(const MeshDev M, const double* __restrict__ v, double* __restrict__ vf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M.n_free) vf[i] = v[M.free_nodes[i]];
}

// dL/dkappa_e = -lam_e^T K_e^0 u_e  (K_e^0: element matrix at kappa = 1)
__global__ void k_grad_elem(const MeshDev M, const double* __restrict__ lam, const double* __restrict__ u,
                            double* __restrict__ gk) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= M.n_el) return;
  double g = 0.0;
  if (M.npe != M.dim + 1) {                                 // P2: -lam_e^T K_e^0 u_e with the closed-form K_e^0
    if (M.dim == 1) {
      const int n[3] = {M.elems[3 * e], M.elems[3 * e + 1], M.elems[3 * e + 2]};
      const double h = M.nodes[n[1]] - M.nodes[n[0]];
      double acc = 0.0;
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) acc = fma(lam[n[i]] * p2_line_k0(i, j), u[n[j]], acc);
      g = -acc / (3.0 * h);
    } else {
      int n[6];
      const P2Tri T = p2_tri_of(M, e, n);
      if (T.keep) {
        double ue[6], acc = 0.0;
#pragma unroll
        for (int j = 0; j < 6; ++j) ue[j] = u[n[j]];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          double kr[6], ri = 0.0;
          p2_tri_k0_row(T, i, kr);
#pragma unroll
          for (int j = 0; j < 6; ++j) ri = fma(kr[j], ue[j], ri);
          acc = fma(lam[n[i]], ri, acc);
        }
        g = -acc;
      }
    }
  } else if (M.dim == 1) {
    const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
    const double h = M.nodes[j] - M.nodes[i];
    g = -(lam[j] - lam[i]) * (u[j] - u[i]) / h;
  } else {
    int n[3];
    const Elem2D E = elem2d(M, e, n);
    if (!(E.area < AREA_EPS)) {
      double bl = 0, bu = 0, cl = 0, cu = 0;
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const double l = lam[n[q]], uu = u[n[q]];
        bl = fma(E.b[q], l, bl);
        bu = fma(E.b[q], uu, bu);
        cl = fma(E.c[q], l, cl);
        cu = fma(E.c[q], uu, cu);
      }
      g = -(bl * bu + cl * cu) / (4.0 * E.area);
    }
  }
  gk[e] = g;
}

// dL/df: 1-D  gf_p = sum_{e∋p} (h_e/2) lam_p ;  2-D  gf_q = sum_{e∋q} (area_e/9) sum_{p∈e} lam_p
__global__ void k_grad_f(const MeshDev M, const double* __restrict__ lam, double* __restrict__ gf) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_nodes) return;
  double g = 0.0;
  for (int a = M.adj_ptr[p]; a < M.adj_ptr[p + 1]; ++a) {
    const int e = M.adj_elem[a];
    if (M.npe != M.dim + 1) {                               // P2: dL/df = M lam (consistent mass, symmetric)
      const int loc = M.adj_loc[a];
      if (M.dim == 1) {
        const int n[3] = {M.elems[3 * e], M.elems[3 * e + 1], M.elems[3 * e + 2]};
        double r = 0.0;
#pragma unroll
        for (int q = 0; q < 3; ++q) r = fma(p2_line_m(loc, q), lam[n[q]], r);
        g = fma((M.nodes[n[1]] - M.nodes[n[0]]) / 30.0, r, g);
      } else {
        int n[6];
        const P2Tri T = p2_tri_of(M, e, n);
        if (!T.keep) continue;
        double mr[6], r = 0.0;
        p2_tri_m_row(loc, mr);
#pragma unroll
        for (int q = 0; q < 6; ++q) r = fma(mr[q], lam[n[q]], r);
        g = fma(T.area * (1.0 / 180.0), r, g);
      }
    } else if (M.dim == 1) {
      const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
      g = fma((M.nodes[j] - M.nodes[i]) * 0.5, lam[p], g);
    } else {
      int n[3];
      const Elem2D E = elem2d(M, e, n);
      if (E.area < AREA_EPS) continue;
      g = fma(E.area / 9.0, (lam[n[0]] + lam[n[1]]) + lam[n[2]], g);
    }
  }
  gf[p] = g;
}

// deterministic sum of n doubles by ONE block (fixed order for a fixed n)
__global__ void k_sum(const double* __restrict__ in, long long n, double* __restrict__ out) {
  __shared__ double sh[1024];
  double a = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) a += in[i];
  sh[threadIdx.x] = a;
  __syncthreads();
  for (int d = blockDim.x / 2; d > 0; d >>= 1) {
    if (static_cast<int>(threadIdx.x) < d) sh[threadIdx.x] += sh[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
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
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}
void leave(const dfe_mesh* m, int prev) {
  if (prev != m->info.device) cudaSetDevice(prev);
}
int check_launch(const char* who) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    dfe::set_error("%s: kernel launch failed: %s", who, cudaGetErrorString(e));
    return DFE_ERR_CUDA;
  }
  return DFE_OK;
}
inline unsigned blocks(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

}  // namespace

extern "C" int dfe_assemble(const dfe_mesh* m, const double* kappa, int kappa_mode, const double* f,
                            double* vals_full, double* F, void* stream) {
  int prev;
  int rc = enter(m, "dfe_assemble", &prev);
  if (rc) return rc;
  if (!kappa || !f || !vals_full || !F) {
    dfe::set_error("dfe_assemble: null argument");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_SCALAR && kappa_mode != DFE_KAPPA_PER_ELEMENT) {
    dfe::set_error("dfe_assemble: kappa_mode must be SCALAR or PER_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else {
    // A/B switches, read per call so that the tests can compare the three kernels bit for bit in one process
    const bool no_grid = getenv("DFE_ASSEMBLE_GENERAL") != nullptr;   // general kernel on structured meshes
    const bool row_grid = getenv("DFE_ASSEMBLE_ROWS") != nullptr;     // row-owner structured kernel
    const bool k16 = (reinterpret_cast<uintptr_t>(kappa) & 15) == 0;         // per-element kappa is read as pairs
    if (m->topo_nx > 0 && !no_grid && !row_grid && k16) {
      const dim3 grid(blocks(m->topo_nx + 1, AN_C), blocks(m->topo_ny + 1, AN_R));
      const int pe = kappa_mode == DFE_KAPPA_PER_ELEMENT;
      cudaStream_t st = static_cast<cudaStream_t>(stream);
      if (m->topo_geo_mid) {   // geometry range verified at handle creation: only kappa and the load sum are checked per call
        cudaFuncSetAttribute(k_assemble_tile<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        k_assemble_tile<true><<<grid, AQ_T, 0, st>>>(m->dev, m->topo_nx, m->topo_ny, kappa, pe, f, vals_full, F);
      } else {
        cudaFuncSetAttribute(k_assemble_tile<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        k_assemble_tile<false><<<grid, AQ_T, 0, st>>>(m->dev, m->topo_nx, m->topo_ny, kappa, pe, f, vals_full, F);
      }
    } else if (m->topo_nx > 0 && !no_grid)
      k_assemble_grid<<<blocks(m->dev.n_nodes, AG_T), AG_T, 0, static_cast<cudaStream_t>(stream)>>>(
          m->dev, m->topo_nx, m->topo_ny, kappa, kappa_mode == DFE_KAPPA_PER_ELEMENT, f, vals_full, F);
    else
      k_assemble<<<blocks(m->dev.n_nodes, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
          m->dev, kappa, kappa_mode == DFE_KAPPA_PER_ELEMENT, f, vals_full, F);
    rc = check_launch("dfe_assemble");
  }
  leave(m, prev);
  return rc;
}

extern "C" int dfe_eliminate(const dfe_mesh* m, const double* vals_full, const double* F, double* vals_free,
                             double* sell_vals, double* F_free, double* dinv, void* stream) {
  int prev;
  int rc = enter(m, "dfe_eliminate", &prev);
  if (rc) return rc;
  if (!vals_full || !F || !F_free || !dinv) {
    dfe::set_error("dfe_eliminate: null argument");
    rc = DFE_ERR_INVALID;
  } else if (m->dev.n_free > 0) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    k_eliminate<<<blocks(m->dev.n_free, 128), 128, 0, st>>>(m->dev, vals_full, F, vals_free, F_free, dinv);
    if (sell_vals)
      k_fill_sell<<<blocks(m->dev.sell_nnz, 256) < 4096u ? blocks(m->dev.sell_nnz, 256) : 4096u, 256, 0, st>>>(
          m->dev, vals_full, sell_vals);
    rc = check_launch("dfe_eliminate");
  }
  leave(m, prev);
  return rc;
}

extern "C" int dfe_scatter(const dfe_mesh* m, const double* x_free, int zero_bc, double* u, void* stream) {
  int prev;
  int rc = enter(m, "dfe_scatter", &prev);
  if (rc) return rc;
  if (!u || (!x_free && m->dev.n_free > 0)) {
    dfe::set_error("dfe_scatter: null argument");
    rc = DFE_ERR_INVALID;
  } else {
    const int n = m->dev.n_free > m->dev.n_dir ? m->dev.n_free : m->dev.n_dir;
    k_scatter<<<blocks(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(m->dev, x_free, zero_bc, u);
    rc = check_launch("dfe_scatter");
  }
  leave(m, prev);
  return rc;
}

extern "C" int dfe_gather_free(const dfe_mesh* m, const double* v_full, double* v_free, void* stream) {
  int prev;
  int rc = enter(m, "dfe_gather_free", &prev);
  if (rc) return rc;
  if (!v_full || (!v_free && m->dev.n_free > 0)) {
    dfe::set_error("dfe_gather_free: null argument");
    rc = DFE_ERR_INVALID;
  } else if (m->dev.n_free > 0) {
    k_gather<<<blocks(m->dev.n_free, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(m->dev, v_full, v_free);
    rc = check_launch("dfe_gather_free");
  }
  leave(m, prev);
  return rc;
}

extern "C" size_t dfe_grad_workspace_bytes(const dfe_mesh* m) {
  return m ? (static_cast<size_t>(m->info.n_elements) + 32) * sizeof(double) : 0;
}

extern "C" int dfe_grad(const dfe_mesh* m, const double* lam_full, const double* u, const double* kappa,
                        int kappa_mode, double* gkappa, double* gf, void* ws, size_t ws_bytes, void* stream) {
  (void)kappa;  // K is linear in kappa: K_e = kappa_e K_e^0, the gradient does not need its value
  int prev;
  int rc = enter(m, "dfe_grad", &prev);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!lam_full || !u || !gkappa) {
    dfe::set_error("dfe_grad: null argument");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode == DFE_KAPPA_PER_ELEMENT) {
    if (m->dev.n_el > 0) k_grad_elem<<<blocks(m->dev.n_el, 256), 256, 0, st>>>(m->dev, lam_full, u, gkappa);
  } else if (kappa_mode == DFE_KAPPA_SCALAR) {
    if (!ws || ws_bytes < dfe_grad_workspace_bytes(m)) {
      dfe::set_error("dfe_grad: workspace too small");
      rc = DFE_ERR_WORKSPACE;
    } else {
      double* tmp = static_cast<double*>(ws);
      if (m->dev.n_el > 0) k_grad_elem<<<blocks(m->dev.n_el, 256), 256, 0, st>>>(m->dev, lam_full, u, tmp);
      k_sum<<<1, 1024, 0, st>>>(tmp, m->dev.n_el, gkappa);
    }
  } else {
    dfe::set_error("dfe_grad: kappa_mode must be SCALAR or PER_ELEMENT");
    rc = DFE_ERR_INVALID;
  }
  if (rc == DFE_OK && gf) k_grad_f<<<blocks(m->dev.n_nodes, 128), 128, 0, st>>>(m->dev, lam_full, gf);
  if (rc == DFE_OK) rc = check_launch("dfe_grad");
  leave(m, prev);
  return rc;
}
