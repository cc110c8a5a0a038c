// P1 / P2 row-owner assembly shared by dfe_general.cu (dfe_assemble) and dfe_band_ps.cu (the per-sample matrices of the
// batched banded route), included inside an anonymous namespace after `using dfe::MeshDev;`.  One definition keeps the
// assembled values of both routes bit-identical.
#pragma once

constexpr double AREA_EPS = 1e-15;  // solver.py:120

#include "dfe_p2.cuh"   // closed-form P2 element matrices (roadmap extension, no upstream arithmetic)

// vertices of P2 triangle e (the first three of its six nodes)
__device__ __forceinline__ P2Tri p2_tri_of(const MeshDev& M, int e, int (&n)[6]) {
#pragma unroll
  for (int q = 0; q < 6; ++q) n[q] = M.elems[6 * e + q];
  const double x[3] = {M.nodes[2 * n[0]], M.nodes[2 * n[1]], M.nodes[2 * n[2]]};
  const double y[3] = {M.nodes[2 * n[0] + 1], M.nodes[2 * n[1] + 1], M.nodes[2 * n[2] + 1]};
  return p2_tri_geom(x, y);
}

struct Elem2D {
  double area, b[3], c[3];
};

// solver.py:114-134 in the reference's operation order
__device__ __forceinline__ Elem2D elem2d(const MeshDev& M, int e, int n[3]) {
  n[0] = M.elems[3 * e + 0];
  n[1] = M.elems[3 * e + 1];
  n[2] = M.elems[3 * e + 2];
  const double xi = M.nodes[2 * n[0]], yi = M.nodes[2 * n[0] + 1];
  const double xj = M.nodes[2 * n[1]], yj = M.nodes[2 * n[1] + 1];
  const double xk = M.nodes[2 * n[2]], yk = M.nodes[2 * n[2] + 1];
  Elem2D E;
  const double t1 = __dmul_rn(__dsub_rn(xj, xi), __dsub_rn(yk, yi));
  const double t2 = __dmul_rn(__dsub_rn(xk, xi), __dsub_rn(yj, yi));
  E.area = __dmul_rn(0.5, fabs(__dsub_rn(t1, t2)));
  E.b[0] = __dsub_rn(yj, yk);
  E.b[1] = __dsub_rn(yk, yi);
  E.b[2] = __dsub_rn(yi, yj);
  E.c[0] = __dsub_rn(xk, xj);
  E.c[1] = __dsub_rn(xi, xk);
  E.c[2] = __dsub_rn(xj, xi);
  return E;
}

// Row-owner assembly for arbitrary meshes.  The row is accumulated in a thread-local array (rows of up to ROWMAX
// structural entries — every P1 mesh of reasonable quality) and written once; wider rows fall back to read-modify-write
// in global memory.  Both orders of additions are the reference's.  LOAD = false assembles the matrix row alone (f and F
// are not touched and may be null).
constexpr int ROWMAX = 16;

template <bool LOCAL, bool LOAD = true>
__device__ __forceinline__ void assemble_row(const MeshDev& M, int p, const double* __restrict__ kappa, int per_elem,
                                             const double* __restrict__ f, double* __restrict__ vals, double* __restrict__ F) {
  const int r0 = M.rowptr[p], r1 = M.rowptr[p + 1];
  double acc[ROWMAX];
  if (LOCAL) {
#pragma unroll
    for (int k = 0; k < ROWMAX; ++k) acc[k] = 0.0;
  } else {
    for (int k = r0; k < r1; ++k) vals[k] = 0.0;
  }
  auto add = [&](int slot, double v) {
    if (LOCAL) acc[slot - r0] = __dadd_rn(acc[slot - r0], v);
    else vals[slot] = __dadd_rn(vals[slot], v);
  };
  double Fp = 0.0;
  for (int a = M.adj_ptr[p]; a < M.adj_ptr[p + 1]; ++a) {
    const int e = M.adj_elem[a];
    const int loc = M.adj_loc[a];
    const double kap = kappa[per_elem ? e : 0];
    if (M.npe != M.dim + 1) {                               // P2 (dfe_p2.cuh); F = M f with the consistent mass matrix
      if (M.dim == 1) {
        const int n[3] = {M.elems[3 * e], M.elems[3 * e + 1], M.elems[3 * e + 2]};
        const double h = M.nodes[n[1]] - M.nodes[n[0]];
        const double ks = kap / (3.0 * h), ms = h / 30.0;
        double fl = 0.0;
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          add(M.adj_slot[3 * a + q], ks * p2_line_k0(loc, q));
          if (LOAD) fl = fma(p2_line_m(loc, q), f[n[q]], fl);
        }
        if (LOAD) Fp = fma(ms, fl, Fp);
      } else {
        int n[6];
        const P2Tri T = p2_tri_of(M, e, n);
        if (!T.keep) continue;
        double kr[6], mr[6];
        p2_tri_k0_row(T, loc, kr);
        p2_tri_m_row(loc, mr);
        double fl = 0.0;
#pragma unroll
        for (int q = 0; q < 6; ++q) {
          add(M.adj_slot[6 * a + q], kap * kr[q]);
          if (LOAD) fl = fma(mr[q], f[n[q]], fl);
        }
        if (LOAD) Fp = fma(T.area * (1.0 / 180.0), fl, Fp);
      }
    } else if (M.dim == 1) {
      const int i = M.elems[2 * e], j = M.elems[2 * e + 1];
      const double h = __dsub_rn(M.nodes[j], M.nodes[i]);   // solver.py:84-85
      const double ke = __ddiv_rn(kap, h);                  // :88
      // row `loc` of k_e [[1,-1],[-1,1]]  (:89-92: K[i,i]+k, K[i,j]-k, K[j,i]-k, K[j,j]+k)
      const int s0 = M.adj_slot[2 * a], s1 = M.adj_slot[2 * a + 1];
      add(s0, loc == 0 ? ke : -ke);                         // x - k == x + (-k) bit for bit
      add(s1, loc == 0 ? -ke : ke);
      if (LOAD) Fp = __dadd_rn(Fp, __dmul_rn(__ddiv_rn(h, 2.0), f[p]));  // :95-96
    } else {
      int n[3];
      const Elem2D E = elem2d(M, e, n);
      if (E.area < AREA_EPS) continue;  // :120-121
      const double den = __dmul_rn(4.0, E.area);
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        // k_pq = kappa*(b_p b_q + c_p c_q)/(4 area)   (:139)
        const double num = __dmul_rn(kap, __dadd_rn(__dmul_rn(E.b[loc], E.b[q]), __dmul_rn(E.c[loc], E.c[q])));
        add(M.adj_slot[3 * a + q], __ddiv_rn(num, den));
      }
      // F_p += area/3 * (f_i+f_j+f_k)/3   (:143-145)
      if (LOAD) {
        const double fc = __ddiv_rn(__dadd_rn(__dadd_rn(f[n[0]], f[n[1]]), f[n[2]]), 3.0);
        Fp = __dadd_rn(Fp, __dmul_rn(__ddiv_rn(E.area, 3.0), fc));
      }
    }
  }
  if (LOAD) F[p] = Fp;
  if (LOCAL)
    for (int k = r0; k < r1; ++k) vals[k] = acc[k - r0];
}
