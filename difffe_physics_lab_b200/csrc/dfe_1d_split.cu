// Two-pass ("split") fused 1-D solve / adjoint for chain meshes with exactly one Neumann sweep.
//
// Same mathematics as dfe_1d.cu (K = M + E, x = M^{-1}F - M^{-1}E M^{-1}F, flux-form prefix sums), but the
// cross-CTA dependency of the prefix sums is removed by LINEARITY instead of by an on-chip exchange:
// inside a chunk everything a CTA computes is affine in two scalars that depend on the other chunks,
//
//   x0_i = alpha + beta * Xl_i - W0l_i           (Xl, W0l: prefix sums from the chunk's first node)
//   rhs1_i = -delta_i x0_i = alpha*err_i + beta*(err_i Xl_i) - err_i W0l_i
//
// so pass 1 publishes, per (sample, chunk), the stage-0 summary and the summaries of the three component
// vectors (err, err*Xl, err*W0l) — 12-16 doubles; a tiny fold kernel (one warp per sample) turns them into
// (alpha, beta) and the stage-1 pair (alpha1, beta1) for every chunk (and, backward, finishes dL/dkappa);
// pass 2 re-reads the row chunk and writes u = x0 + x1 (or dL/df) directly.
//
// Trade: the input row is read twice (24 B/node forward instead of 16 B/node — the second read is served
// by the 126 MB L2 when the batch is walked in L2-sized slabs), in exchange for CTAs that never wait for
// each other: no co-residency requirement, any mesh size, any batch size, plain streaming occupancy.
// CTA c of a column always owns chunk c of the mesh (element data stay in shared memory for the whole
// batch); rows move with 1-D TMA bulk copies, double-buffered.
#include <cstdint>
#include <cstdlib>

#include "dfe_internal.h"

namespace {

#include "dfe_1d_common.cuh"

constexpr int ST = 256;          // threads per CTA
constexpr int SR = 13;           // nodes per thread (odd -> conflict-free LDS.64)
constexpr int SCH = SR * ST;     // chunk capacity (3328 nodes)
constexpr int SNW = ST / 32;
constexpr int NP1 = 16;          // doubles per (sample, chunk) written by pass 1
constexpr int NP2 = 4;           // doubles per (sample, chunk) read by pass 2: alpha, beta, alpha1, beta1

struct PS {
  int nn, G, chg, NG;
  long long B, s_begin, s_end;   // this launch covers samples [s_begin, s_end)
  const double* hs;      // global: h_e/2
  const double* rh;      // global: RN(1/(h_e/2))
  const double* in0;     // forward: f ; backward: gbar
  long long ld0;
  const double* in1;     // backward: u
  long long ld1;
  double* out;           // forward: u ; backward: dL/df (may be null -> pass 2 is skipped)
  long long ldo;
  const double* kappa;
  int per_sample;
  int bcL, bcR;
  double gL, gR;
  double* part;          // [B][G][NP1]
  double* coef;          // [B][G][NP2]
  double* gk;            // backward, scalar kappa: [B] per-sample dL/dkappa
  // per-element kappa (PE kernels): kappa row of sample s = kap_row + s*ldk (ldk = 0: field shared by the batch)
  const double* kap_row;
  long long ldk;
  double* gke_out;       // backward PE, per-sample field: (B, n_el) output rows
  double* gk_cols;       // backward PE, shared field: [NG][n_el] per-column partial sums
  int sup0, sup1, supk;  // PE kernels: in0 / in1 / kap_row start on a 16-byte boundary (aligned-superset row loads)
};

// chunk-static bookkeeping shared by both passes
struct Chunk {
  int n0, len, tb, nin, nst;
  bool ownsL, ownsR;
};
__device__ __forceinline__ Chunk make_chunk(const PS& p, int c, int tid) {
  Chunk k;
  k.n0 = c * p.chg;
  const int n1 = min(p.nn, k.n0 + p.chg);
  k.len = n1 - k.n0;
  k.tb = tid * SR;
  k.nin = max(0, min(SR, min(k.len, p.nn - (p.bcR ? 1 : 0) - k.n0) - k.tb));
  k.nst = max(0, min(SR, k.len - k.tb));
  k.ownsL = p.bcL && c == 0 && tid == 0;
  k.ownsR = p.bcR && c == p.G - 1 && tid == (k.len - 1) / SR;
  return k;
}
__device__ __forceinline__ void load_mesh_chunk(const PS& p, const Chunk& k, double* hsS, double* rhS, int tid) {
  for (int j = tid; j <= SCH; j += ST) {
    const int e = k.n0 - 1 + j;
    const bool ex = (e >= 0 && e < p.nn - 1 && j <= k.len);
    hsS[j] = ex ? p.hs[e] : 0.0;
    rhS[j] = ex ? p.rh[e] : 0.0;
  }
}

// thread 0: start the bulk load of one row chunk (plus the unaligned head/tail elements)
__device__ __forceinline__ void issue_row(double* sbuf, const double* g, int len, uint64_t* bar, uint32_t extra_bytes) {
  const Seg q = make_seg(g, len);
  if (q.head) sbuf[q.mis] = g[0];
  if (q.tail) sbuf[q.mis + len - 1] = g[len - 1];
  mbar_arrive_expect_tx(bar, 8u * static_cast<uint32_t>(q.body) + extra_bytes);
  if (q.body) bulk_g2s(sbuf + q.mis + q.head, g + q.head, 8u * q.body, bar);
}
__device__ __forceinline__ int mis_of(const double* g) {
  return static_cast<int>((reinterpret_cast<uintptr_t>(g) >> 3) & 1);
}

// Row loads of the per-element kernels (thread 0).  [g, g + len) goes to sbuf with element j at sbuf[mis + j].  When the
// array starts on a 16-byte boundary (`sup`) the 16-byte aligned SUPERSET [g - mis, ...) is fetched with one bulk copy: the
// element before / after the range belongs to the same array, except past its very last element (`last`).  Otherwise the
// unaligned head / tail elements are fetched by scalar loads — which stall thread 0 for a DRAM latency before it can start
// the bulk copy (measured: the exposed part of every sample in the round-1 version of these kernels).
__device__ __forceinline__ uint32_t row_tx_bytes(const double* g, int len, bool sup, bool last) {
  if (len <= 0) return 0u;
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g) >> 3) & 1);
  if (sup) {
    int cnt = (mis + len + 1) & ~1;
    if (last && ((mis + len) & 1)) cnt -= 2;
    return 8u * static_cast<uint32_t>(cnt);
  }
  return 8u * static_cast<uint32_t>(make_seg(g, len).body);
}
__device__ __forceinline__ void row_scalars(double* sbuf, const double* g, int len, bool sup, bool last) {
  if (len <= 0) return;
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g) >> 3) & 1);
  if (sup) {
    if (last && ((mis + len) & 1)) sbuf[mis + len - 1] = g[len - 1];
  } else {
    const Seg q = make_seg(g, len);
    if (q.head) sbuf[q.mis] = g[0];
    if (q.tail) sbuf[q.mis + len - 1] = g[len - 1];
  }
}
__device__ __forceinline__ void row_bulk(double* sbuf, const double* g, int len, bool sup, bool last, uint64_t* bar) {
  if (len <= 0) return;
  const int mis = static_cast<int>((reinterpret_cast<uintptr_t>(g) >> 3) & 1);
  if (sup) {
    int cnt = (mis + len + 1) & ~1;
    if (last && ((mis + len) & 1)) cnt -= 2;
    if (cnt > 0) bulk_g2s(sbuf, g - mis, 8u * cnt, bar);
  } else {
    const Seg q = make_seg(g, len);
    if (q.body) bulk_g2s(sbuf + q.mis + q.head, g + q.head, 8u * q.body, bar);
  }
}

// CTA-level exclusive prefix of per-thread triples.  Two-level: warp shuffle scan, then every warp scans
// the SNW warp totals with 3 more shuffle steps (cheaper than a serial fold in every thread).
// `tot` = CTA total, valid in every thread.
__device__ __forceinline__ Tri cta_excl_scan(const Tri& t, Tri* wt, int lane, int warp, Tri& tot) {
  const Tri inc = warp_incl_scan(t, lane);
  if (lane == 31) wt[warp] = inc;
  __syncthreads();
  Tri x = (lane < SNW) ? wt[lane] : tri_id();
#pragma unroll
  for (int d = 1; d < SNW; d <<= 1) {
    const Tri o = shfl_up_tri(x, d);
    if (lane >= d) x = combine(o, x);
  }
  tot = shfl_tri(x, SNW - 1);
  Tri wc = shfl_tri(x, warp > 0 ? warp - 1 : 0);
  if (warp == 0) wc = tri_id();
  Tri ex = shfl_up_tri(inc, 1);
  if (lane == 0) ex = tri_id();
  return combine(wc, ex);
}

// k_i = fl(kappa/h_i) from the stored reciprocal (Markstein correction: correctly rounded)
__device__ __forceinline__ double kdiv(double kaph, double h, double y) {
  const double q0 = kaph * y;
  return fma(fma(-h, q0, kaph), y, q0);
}
// err = (a + b) - fl(a + b), exact (TwoSum)
__device__ __forceinline__ double two_sum_err(double a, double b) {
  const double d = __dadd_rn(a, b);
  const double bb = __dsub_rn(d, a);
  return __dadd_rn(__dsub_rn(a, __dsub_rn(d, bb)), __dsub_rn(b, bb));
}

// ------------------------------------------------------------------------------------------------ pass 1
// smem: bars | wt | red | hsS | rhS | rows
template <bool BWD>
__global__ void __launch_bounds__(ST, 2) k1d_pass1(const PS p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);               // [2]
  Tri* wt = reinterpret_cast<Tri*>(smem_raw + 64);                     // [SNW]
  double* red = reinterpret_cast<double*>(smem_raw + 64 + SNW * 24);   // [SNW][12]
  double* hsS = reinterpret_cast<double*>(smem_raw + 2048);
  double* rhS = hsS + (SCH + 2);
  double* rows = rhS + (SCH + 2);                                      // FWD: f x2 ; BWD: gbar, u
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x % p.G, col = blockIdx.x / p.G;
  const Chunk ck = make_chunk(p, c, tid);
  load_mesh_chunk(p, ck, hsS, rhS, tid);
  if (tid == 0) {
    mbar_init_raw(bar, 1);
    mbar_init_raw(bar + 1, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const double* hsT = hsS + ck.tb;
  const double* rhT = rhS + ck.tb;

  auto issue = [&](long long s, int b) {
    double* r0 = rows + (BWD ? 0 : b) * (SCH + 4);
    if (BWD) {
      double* r1 = rows + (SCH + 4);
      const double* g1 = p.in1 + s * p.ld1 + ck.n0;
      const Seg q1 = make_seg(g1, ck.len);
      if (q1.head) r1[q1.mis] = g1[0];
      if (q1.tail) r1[q1.mis + ck.len - 1] = g1[ck.len - 1];
      issue_row(r0, p.in0 + s * p.ld0 + ck.n0, ck.len, bar + b, 8u * q1.body);
      if (q1.body) bulk_g2s(r1 + q1.mis + q1.head, g1 + q1.head, 8u * q1.body, bar + b);
    } else {
      issue_row(r0, p.in0 + s * p.ld0 + ck.n0, ck.len, bar + b, 0);
    }
  };

  long long s = p.s_begin + col;
  if (tid == 0 && s < p.s_end) issue(s, 0);
  int it = 0;
  for (; s < p.s_end; s += p.NG, ++it) {
    const int b = BWD ? 0 : (it & 1);
    if (!BWD && tid == 0 && s + p.NG < p.s_end) issue(s + p.NG, b ^ 1);   // prefetch (its buffer was consumed last iteration)
    const double kap = p.kappa[p.per_sample ? s : 0];
    const double kaph = 0.5 * kap, invk2 = 2.0 / kap;
    const double* r0 = rows + (BWD ? 0 : b) * (SCH + 4) + mis_of(p.in0 + s * p.ld0 + ck.n0) + ck.tb;
    const double* r1 = BWD ? rows + (SCH + 4) + mis_of(p.in1 + s * p.ld1 + ck.n0) + ck.tb : nullptr;
    mbar_wait(bar + b, BWD ? (it & 1) : ((it >> 1) & 1));

    // ---- sweep 1: right-hand side and the thread's local triple
    double v[SR];
    Tri t = tri_id();
    {
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < SR; ++j) {
        const double hi = hsT[j + 1];
        const double in = (j < ck.nin) ? r0[j] : 0.0;
        double v0 = BWD ? in : __dadd_rn(__dmul_rn(hp, in), __dmul_rn(hi, in));   // solver.py:95-96
        if (j == 0 && ck.ownsL) v0 = 0.0;
        v[j] = v0;
        const double w = hi * invk2;
        t.s += v0;
        t.w = fma(w, t.s, t.w);
        t.x += w;
        hp = hi;
      }
    }
    Tri tot0;
    const Tri ex = cta_excl_scan(t, wt, lane, warp, tot0);
    // ---- sweep 2: component vectors err, err*Xl, err*W0l: sums A, running sums a, weighted sums Bw
    double S = ex.s, X = ex.x, W = ex.w;
    double a1 = 0, a2 = 0, a3 = 0, B1 = 0, B2 = 0, B3 = 0, D0 = 0, E1 = 0, E2 = 0, E3 = 0, Xt = 0;
    double kp = kdiv(kaph, hsT[0], rhT[0]);
#pragma unroll
    for (int j = 0; j < SR; ++j) {
      const double hi = hsT[j + 1];
      const double ki = kdiv(kaph, hi, rhT[j + 1]);
      const double err = two_sum_err(kp, ki);   // 0 on Dirichlet and padding rows (one k is 0)
      kp = ki;
      S += v[j];
      const double c1 = err, c2 = err * X, c3 = err * W;
      a1 += c1;
      a2 += c2;
      a3 += c3;
      if (BWD) {
        const double uj = (j < ck.nst) ? r1[j] : 0.0;
        D0 = fma(v[j], uj, D0);
        E1 = fma(c1, uj, E1);
        E2 = fma(c2, uj, E2);
        E3 = fma(c3, uj, E3);
      }
      const double w = hi * invk2;
      B1 = fma(w, a1, B1);
      B2 = fma(w, a2, B2);
      B3 = fma(w, a3, B3);
      W = fma(w, S, W);
      X += w;
      Xt += w;
    }
    // ---- CTA totals of the three component triples (ordered combine) and of the plain sums
    // B_total = sum_t [ B_t + (sum_{t'<t} a_t') * Xt_t ]: exclusive prefix of a over threads, then plain sums.
    double p1 = a1, p2 = a2, p3 = a3;   // inclusive warp prefixes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double o1 = __shfl_up_sync(0xffffffffu, p1, d), o2 = __shfl_up_sync(0xffffffffu, p2, d),
                   o3 = __shfl_up_sync(0xffffffffu, p3, d);
      if (lane >= d) { p1 += o1; p2 += o2; p3 += o3; }
    }
    // warp-local: Bw = sum_lanes [B + (excl prefix within warp)*Xt]; cross-warp part added by thread 0 below
    double q1 = fma(p1 - a1, Xt, B1), q2 = fma(p2 - a2, Xt, B2), q3 = fma(p3 - a3, Xt, B3), xw = Xt;
    double e0 = D0, e1 = E1, e2 = E2, e3 = E3;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      q1 += __shfl_xor_sync(0xffffffffu, q1, d);
      q2 += __shfl_xor_sync(0xffffffffu, q2, d);
      q3 += __shfl_xor_sync(0xffffffffu, q3, d);
      xw += __shfl_xor_sync(0xffffffffu, xw, d);
      if (BWD) {
        e0 += __shfl_xor_sync(0xffffffffu, e0, d);
        e1 += __shfl_xor_sync(0xffffffffu, e1, d);
        e2 += __shfl_xor_sync(0xffffffffu, e2, d);
        e3 += __shfl_xor_sync(0xffffffffu, e3, d);
      }
    }
    if (lane == 31) {
      double* r = red + warp * 12;
      r[0] = p1; r[1] = p2; r[2] = p3;       // warp sums of a
      r[3] = q1; r[4] = q2; r[5] = q3;       // warp-local weighted sums
      r[6] = xw;                             // warp X length
      r[7] = e0; r[8] = e1; r[9] = e2; r[10] = e3;
    }
    __syncthreads();
    if (tid == 0) {
      double A1 = 0, A2 = 0, A3 = 0, Q1 = 0, Q2 = 0, Q3 = 0, d0 = 0, f1 = 0, f2 = 0, f3 = 0;
      for (int w = 0; w < SNW; ++w) {
        const double* r = red + w * 12;
        Q1 += fma(A1, r[6], r[3]);           // warps before w contribute (sum a) * X_w
        Q2 += fma(A2, r[6], r[4]);
        Q3 += fma(A3, r[6], r[5]);
        A1 += r[0]; A2 += r[1]; A3 += r[2];
        d0 += r[7]; f1 += r[8]; f2 += r[9]; f3 += r[10];
      }
      double* o = p.part + (s * p.G + c) * NP1;
      o[0] = tot0.s; o[1] = tot0.x; o[2] = tot0.w;
      o[3] = A1; o[4] = Q1; o[5] = A2; o[6] = Q2; o[7] = A3; o[8] = Q3;
      o[9] = d0; o[10] = f1; o[11] = f2; o[12] = f3;
    }
    __syncthreads();   // red / wt / the single backward row buffer are reused by the next sample
    if (BWD && tid == 0 && s + p.NG < p.s_end) issue(s + p.NG, 0);
  }
}

// ------------------------------------------------------------------------------------------------ fold
// One warp per sample: prefix over the G chunk summaries for stage 0 and stage 1, chunk coefficients, dL/dkappa.
template <bool BWD>
__global__ void k1d_fold(const PS p) {
  const int lane = threadIdx.x & 31;
  const long long s = p.s_begin + (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
  if (s >= p.s_end) return;
  const int G = p.G;
  const double* part = p.part + s * G * NP1;
  double* coef = p.coef + s * G * NP2;
  const bool LR = p.bcL && p.bcR;
  // ---- stage-0 totals
  Tri base = tri_id();
  for (int g0 = 0; g0 < G; g0 += 32) {
    const int g = g0 + lane;
    Tri t = tri_id();
    if (g < G) { t.s = part[g * NP1]; t.x = part[g * NP1 + 1]; t.w = part[g * NP1 + 2]; }
    t = combine(base, warp_incl_scan(t, lane));
    base = shfl_tri(t, 31);
  }
  const Tri tot0 = base;
  double C0, x0c;
  if (LR) { x0c = 0.0; C0 = tot0.w / tot0.x; }
  else if (p.bcL) { x0c = 0.0; C0 = tot0.s; }
  else { C0 = 0.0; x0c = tot0.w; }
  // x_g = M^{-1}(lifted Dirichlet loads) = ga*X + gb (harmonic interpolant), forward only
  const double ga = (!BWD && LR) ? (p.gR - p.gL) / tot0.x : 0.0;
  const double gb = BWD ? 0.0 : (p.bcL ? p.gL : p.gR);
  // ---- per-chunk (alpha, beta), stage-1 summaries and their running prefix
  base = tri_id();
  Tri base1 = tri_id();
  double dotacc = 0.0;
  for (int g0 = 0; g0 < G; g0 += 32) {
    const int g = g0 + lane;
    Tri t = tri_id();
    if (g < G) { t.s = part[g * NP1]; t.x = part[g * NP1 + 1]; t.w = part[g * NP1 + 2]; }
    const Tri inc = combine(base, warp_incl_scan(t, lane));
    Tri ex = shfl_up_tri(inc, 1);
    if (lane == 0) ex = base;
    base = shfl_tri(inc, 31);
    double alpha = 0.0, beta = 0.0;
    Tri t1 = tri_id();
    if (g < G) {
      const double* q = part + g * NP1;
      alpha = (x0c + C0 * ex.x - ex.w) + fma(ga, ex.x, gb);
      beta = (C0 - ex.s) + ga;
      t1.s = alpha * q[3] + beta * q[5] - q[7];
      t1.w = alpha * q[4] + beta * q[6] - q[8];
      t1.x = q[1];
      if (BWD) dotacc += q[9] + (alpha * q[10] + beta * q[11] - q[12]);
      coef[g * NP2] = alpha;
      coef[g * NP2 + 1] = beta;
    }
    const Tri inc1 = combine(base1, warp_incl_scan(t1, lane));
    Tri ex1 = shfl_up_tri(inc1, 1);
    if (lane == 0) ex1 = base1;
    base1 = shfl_tri(inc1, 31);
    if (g < G) {   // park the stage-1 carry-in; finalised below once the stage-1 totals are known
      coef[g * NP2 + 2] = ex1.w;
      coef[g * NP2 + 3] = ex1.s;
    }
  }
  const Tri tot1 = base1;
  double C1, x1c;
  if (LR) { x1c = 0.0; C1 = tot1.w / tot1.x; }
  else if (p.bcL) { x1c = 0.0; C1 = tot1.s; }
  else { C1 = 0.0; x1c = tot1.w; }
  __syncwarp();
  base = tri_id();
  for (int g0 = 0; g0 < G; g0 += 32) {
    const int g = g0 + lane;
    Tri t = tri_id();
    if (g < G) t.x = part[g * NP1 + 1];
    const Tri inc = combine(base, warp_incl_scan(t, lane));
    Tri ex = shfl_up_tri(inc, 1);
    if (lane == 0) ex = base;
    base = shfl_tri(inc, 31);
    if (g < G) {
      const double w1in = coef[g * NP2 + 2], s1in = coef[g * NP2 + 3];
      coef[g * NP2 + 2] = x1c + C1 * ex.x - w1in;   // alpha1
      coef[g * NP2 + 3] = C1 - s1in;                // beta1
    }
  }
  if (BWD && p.gk != nullptr) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) dotacc += __shfl_xor_sync(0xffffffffu, dotacc, d);
    if (lane == 0) {
      // dL/dkappa = -(1/kappa) sum_stages [ sum_i rhs_i u_i + C (u_R - u_L) - S_tot u_R ]
      const double uL = p.in1[s * p.ld1], uR = p.in1[s * p.ld1 + p.nn - 1];
      const double kap = p.kappa[p.per_sample ? s : 0];
      const double bnd = (C0 + C1) * (uR - uL) - (tot0.s + tot1.s) * uR;
      p.gk[s] = -(dotacc + bnd) / kap;
    }
  }
}

// ------------------------------------------------------------------------------------------------ pass 2
template <bool BWD>
__global__ void __launch_bounds__(ST, 2) k1d_pass2(const PS p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);               // [2]
  Tri* wt = reinterpret_cast<Tri*>(smem_raw + 64);                     // [2][SNW]
  double* hsS = reinterpret_cast<double*>(smem_raw + 2048);
  double* rhS = hsS + (SCH + 2);
  double* rows = rhS + (SCH + 2);                                      // [2][SCH+4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x % p.G, col = blockIdx.x / p.G;
  const Chunk ck = make_chunk(p, c, tid);
  load_mesh_chunk(p, ck, hsS, rhS, tid);
  if (tid == 0) {
    mbar_init_raw(bar, 1);
    mbar_init_raw(bar + 1, 1);
    fence_mbar_init();
  }
  __syncthreads();
  const double* hsT = hsS + ck.tb;
  const double* rhT = rhS + ck.tb;

  long long s = p.s_begin + col;
  if (tid == 0 && s < p.s_end) issue_row(rows, p.in0 + s * p.ld0 + ck.n0, ck.len, bar, 0);
  int it = 0;
  for (; s < p.s_end; s += p.NG, ++it) {
    const int b = it & 1;
    double* buf = rows + b * (SCH + 4);
    if (tid == 0 && s + p.NG < p.s_end) {
      bulk_wait_read0();   // the store issued from the other buffer last iteration has read it
      issue_row(rows + (b ^ 1) * (SCH + 4), p.in0 + (s + p.NG) * p.ld0 + ck.n0, ck.len, bar + (b ^ 1), 0);
    }
    const double kap = p.kappa[p.per_sample ? s : 0];
    const double kaph = 0.5 * kap, invk2 = 2.0 / kap;
    const double* cf = p.coef + (s * p.G + c) * NP2;
    const double alpha = cf[0], beta = cf[1], alpha1 = cf[2], beta1 = cf[3];
    const int mi = mis_of(p.in0 + s * p.ld0 + ck.n0);
    double* go = p.out + s * p.ldo + ck.n0;
    const int mo = mis_of(go);
    mbar_wait(bar + b, (it >> 1) & 1);

    double v[SR];
    Tri t = tri_id();
    {
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < SR; ++j) {
        const double hi = hsT[j + 1];
        const double in = (j < ck.nin) ? buf[mi + ck.tb + j] : 0.0;
        double v0 = BWD ? in : __dadd_rn(__dmul_rn(hp, in), __dmul_rn(hi, in));
        if (j == 0 && ck.ownsL) v0 = 0.0;
        v[j] = v0;
        const double w = hi * invk2;
        t.s += v0;
        t.w = fma(w, t.s, t.w);
        t.x += w;
        hp = hi;
      }
    }
    Tri tot;
    const Tri ex = cta_excl_scan(t, wt, lane, warp, tot);   // barrier: every thread has read its input run
    // ---- x0 = alpha + beta Xl - W0l (parked in the row buffer at the output's alignment); rhs1 = err*x0
    Tri t1 = tri_id();
    {
      double S = ex.s, X = ex.x, W = ex.w;
      double kp = kdiv(kaph, hsT[0], rhT[0]);
#pragma unroll
      for (int j = 0; j < SR; ++j) {
        const double hi = hsT[j + 1];
        S += v[j];
        const double x0 = fma(beta, X, alpha) - W;
        buf[mo + ck.tb + j] = x0;
        const double ki = kdiv(kaph, hi, rhT[j + 1]);
        const double v1 = __dmul_rn(two_sum_err(kp, ki), x0);
        kp = ki;
        v[j] = v1;
        const double w = hi * invk2;
        W = fma(w, S, W);
        X += w;
        t1.s += v1;
        t1.w = fma(w, t1.s, t1.w);
        t1.x += w;
      }
    }
    const Tri ex1 = cta_excl_scan(t1, wt + SNW, lane, warp, tot);
    // ---- x = x0 + (alpha1 + beta1 Xl - W1l)
    {
      double S = ex1.s, X = ex1.x, W = ex1.w;
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < SR; ++j) {
        const double hi = hsT[j + 1];
        S += v[j];
        const double x1 = fma(beta1, X, alpha1) - W;
        const double w = hi * invk2;
        W = fma(w, S, W);
        X += w;
        if (j < ck.nst) {
          const double xv = buf[mo + ck.tb + j] + x1;
          // forward: u[free] = x (solver.py:180-181); backward: dL/df_i = lambda_i (h_{i-1}/2 + h_i/2)
          buf[mo + ck.tb + j] = BWD ? fma(xv, hp, xv * hi) : xv;
        }
        hp = hi;
      }
    }
    if (ck.ownsL) buf[mo] = BWD ? 0.0 : p.gL;              // u[d] = g (solver.py:177-179); dL/df = 0 there
    if (ck.ownsR) buf[mo + ck.len - 1] = BWD ? 0.0 : p.gR;
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      const Seg qo = make_seg(go, ck.len);
      if (qo.head) go[0] = buf[qo.mis];
      if (qo.tail) go[ck.len - 1] = buf[qo.mis + ck.len - 1];
      if (qo.body) bulk_s2g(go + qo.head, buf + qo.mis + qo.head, 8u * qo.body);
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait_read0();
}


// ================================================================================================ per-element kappa
// Same two passes with kappa_e read per element: k_e = fl(kappa_e/h_e) (solver.py:88 with kappa -> kappa[e]),
// w_e = h_e/kappa_e.  R = 9 nodes per thread; the row buffers (input, kappa, and u in the backward pass 2) are DOUBLE
// buffered: the rows of the next sample are in flight while the current one is processed (round 1 had no prefetch and
// ran at two exposed DRAM latencies per sample).  dL/dkappa_e = -(q0_e + q1_e)(u_{e+1}-u_e)/kappa_e with
// q_e = beta - s_e the flux of lambda in element e (s_e: chunk-local inclusive prefix of the rhs).
constexpr int PR = 9;
constexpr int PCH = PR * ST;   // 2304 nodes per chunk

// Slots of elements that do not exist (element -1 of chunk 0, elements past the chunk) are never read: the row buffers
// hold whatever the last bulk load or gradient staging left there — the neighbouring sample's kappa, a dL/dkappa of an
// earlier sample — and an inf or NaN there would otherwise reach this sample through kdiv(k, 0, 0) = 0 * k.
// e0: element n0-1+tb (kT[0]) exists; element n0+tb+j (kT[j+1]) exists iff j < nev.
struct ChunkP {
  int n0, len, tb, nin, nst, nev, eA, ecnt, koff;
  bool ownsL, ownsR, e0;
};
__device__ __forceinline__ ChunkP make_chunk_pe(const PS& p, int c, int tid) {
  ChunkP k;
  k.n0 = c * p.chg;
  const int n1 = min(p.nn, k.n0 + p.chg);
  k.len = n1 - k.n0;
  k.tb = tid * PR;
  k.nin = max(0, min(PR, min(k.len, p.nn - (p.bcR ? 1 : 0) - k.n0) - k.tb));
  k.nst = max(0, min(PR, k.len - k.tb));
  k.nev = max(0, min(PR, min(k.len, p.nn - 1 - k.n0) - k.tb));   // elements owned (right element of each node)
  k.e0 = k.n0 + k.tb >= 1 && k.tb <= k.len && k.n0 + k.tb <= p.nn - 1;
  k.ownsL = p.bcL && c == 0 && tid == 0;
  k.ownsR = p.bcR && c == p.G - 1 && tid == (k.len - 1) / PR;
  // kappa elements held: e in [eA, eA+ecnt), slot j (element n0-1+j) lives at kS[2 + mk + j + koff]
  k.eA = max(k.n0 - 1, 0);
  const int eB = min(k.n0 + k.len - 1, p.nn - 2);
  k.ecnt = max(0, eB - k.eA + 1);
  k.koff = (k.n0 == 0) ? -1 : 0;
  return k;
}
__device__ __forceinline__ void load_mesh_chunk_pe(const PS& p, const ChunkP& k, double* hsS, double* rhS, int tid) {
  for (int j = tid; j <= PCH; j += ST) {
    const int e = k.n0 - 1 + j;
    const bool ex = (e >= 0 && e < p.nn - 1 && j <= k.len);
    hsS[j] = ex ? p.hs[e] : 0.0;
    rhS[j] = ex ? p.rh[e] : 0.0;
  }
}
// CTA scan for the PE kernels (same as cta_excl_scan; separate name only for readability of the call sites)
#define cta_excl_scan_pe cta_excl_scan

constexpr int PBUF = PCH + 8;   // doubles per row buffer
constexpr size_t smem_pe(int nrows) { return 2048 + sizeof(double) * (2 * (PCH + 2) + 2 * nrows * PBUF); }

template <bool BWD>
__global__ void __launch_bounds__(ST, 2) k1d_pe_pass1(const PS p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  Tri* wt = reinterpret_cast<Tri*>(smem_raw + 64);
  double* red = reinterpret_cast<double*>(smem_raw + 64 + SNW * 24);
  double* hsS = reinterpret_cast<double*>(smem_raw + 2048);
  double* rhS = hsS + (PCH + 2);
  double* rin = rhS + (PCH + 2);        // [2] f / gbar row chunk
  double* kS = rin + 2 * PBUF;          // [2] kappa row chunk
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x % p.G, col = blockIdx.x / p.G;
  const ChunkP ck = make_chunk_pe(p, c, tid);
  load_mesh_chunk_pe(p, ck, hsS, rhS, tid);
  for (int j = tid; j < 2 * PBUF; j += ST) kS[j] = 1.0;   // slots of elements that do not exist stay finite
  if (tid == 0) {
    mbar_init_raw(bar, 1);
    mbar_init_raw(bar + 1, 1);
    fence_mbar_init();
  }
  fence_async_smem();
  __syncthreads();
  const double* hsT = hsS + ck.tb;
  const double* rhT = rhS + ck.tb;
  auto issue = [&](long long s, int b) {   // thread 0: rows of sample s -> buffer set b
    const double* g0 = p.in0 + s * p.ld0 + ck.n0;
    const double* gk = p.kap_row + s * p.ldk + ck.eA;
    const bool l0 = s == p.B - 1 && c == p.G - 1;
    const bool lk = (p.ldk == 0 || s == p.B - 1) && ck.eA + ck.ecnt == p.nn - 1;
    double* rb = rin + b * PBUF;
    double* kb = kS + b * PBUF + 2;
    row_scalars(rb, g0, ck.len, p.sup0, l0);
    row_scalars(kb, gk, ck.ecnt, p.supk, lk);
    mbar_arrive_expect_tx(bar + b, row_tx_bytes(g0, ck.len, p.sup0, l0) + row_tx_bytes(gk, ck.ecnt, p.supk, lk));
    row_bulk(rb, g0, ck.len, p.sup0, l0, bar + b);
    row_bulk(kb, gk, ck.ecnt, p.supk, lk, bar + b);
  };

  int it = 0;
  long long s = p.s_begin + col;
  if (tid == 0 && s < p.s_end) issue(s, 0);
  for (; s < p.s_end; s += p.NG, ++it) {
    const int b = it & 1;
    // the other buffer set was last read in iteration it - 1, which ended with a CTA barrier
    if (tid == 0 && s + p.NG < p.s_end) issue(s + p.NG, b ^ 1);
    const double* g0 = p.in0 + s * p.ld0 + ck.n0;
    const double* gk = p.kap_row + s * p.ldk + ck.eA;
    const double* r0 = rin + b * PBUF + mis_of(g0) + ck.tb;
    const double* kT = kS + b * PBUF + 2 + mis_of(gk) + ck.tb + ck.koff;   // kT[j] = kappa of element n0-1+tb+j
    mbar_wait(bar + b, (it >> 1) & 1);

    double v[PR], wv[PR];
    Tri t = tri_id();
    {
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < PR; ++j) {
        const double hi = hsT[j + 1];
        const double in = (j < ck.nin) ? r0[j] : 0.0;
        double v0 = BWD ? in : __dadd_rn(__dmul_rn(hp, in), __dmul_rn(hi, in));
        if (j == 0 && ck.ownsL) v0 = 0.0;
        v[j] = v0;
        // w_e = h_e/kappa_e (hs = h/2); 2 RN(1/k) == RN(2/k)
        const double w = (j < ck.nev) ? hi * (2.0 * __drcp_rn(kT[j + 1])) : 0.0;
        wv[j] = w;
        t.s += v0;
        t.w = fma(w, t.s, t.w);
        t.x += w;
        hp = hi;
      }
    }
    Tri tot0;
    const Tri ex = cta_excl_scan_pe(t, wt, lane, warp, tot0);
    double S = ex.s, X = ex.x, W = ex.w;
    double a1 = 0, a2 = 0, a3 = 0, B1 = 0, B2 = 0, B3 = 0, Xt = 0;
    double kp = ck.e0 ? kdiv(0.5 * kT[0], hsT[0], rhT[0]) : 0.0;
#pragma unroll
    for (int j = 0; j < PR; ++j) {
      const double ki = (j < ck.nev) ? kdiv(0.5 * kT[j + 1], hsT[j + 1], rhT[j + 1]) : 0.0;
      const double err = two_sum_err(kp, ki);
      kp = ki;
      S += v[j];
      const double c2 = err * X, c3 = err * W;
      a1 += err;
      a2 += c2;
      a3 += c3;
      const double w = wv[j];
      B1 = fma(w, a1, B1);
      B2 = fma(w, a2, B2);
      B3 = fma(w, a3, B3);
      W = fma(w, S, W);
      X += w;
      Xt += w;
    }
    double p1 = a1, p2 = a2, p3 = a3;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double o1 = __shfl_up_sync(0xffffffffu, p1, d), o2 = __shfl_up_sync(0xffffffffu, p2, d),
                   o3 = __shfl_up_sync(0xffffffffu, p3, d);
      if (lane >= d) { p1 += o1; p2 += o2; p3 += o3; }
    }
    double q1 = fma(p1 - a1, Xt, B1), q2 = fma(p2 - a2, Xt, B2), q3 = fma(p3 - a3, Xt, B3), xw = Xt;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      q1 += __shfl_xor_sync(0xffffffffu, q1, d);
      q2 += __shfl_xor_sync(0xffffffffu, q2, d);
      q3 += __shfl_xor_sync(0xffffffffu, q3, d);
      xw += __shfl_xor_sync(0xffffffffu, xw, d);
    }
    if (lane == 31) {
      double* r = red + warp * 12;
      r[0] = p1; r[1] = p2; r[2] = p3; r[3] = q1; r[4] = q2; r[5] = q3; r[6] = xw;
    }
    __syncthreads();
    if (tid == 0) {
      double A1 = 0, A2 = 0, A3 = 0, Q1 = 0, Q2 = 0, Q3 = 0;
      for (int w = 0; w < SNW; ++w) {
        const double* r = red + w * 12;
        Q1 += fma(A1, r[6], r[3]);
        Q2 += fma(A2, r[6], r[4]);
        Q3 += fma(A3, r[6], r[5]);
        A1 += r[0]; A2 += r[1]; A3 += r[2];
      }
      double* o = p.part + (s * p.G + c) * NP1;
      o[0] = tot0.s; o[1] = tot0.x; o[2] = tot0.w;
      o[3] = A1; o[4] = Q1; o[5] = A2; o[6] = Q2; o[7] = A3; o[8] = Q3;
      o[9] = 0.0; o[10] = 0.0; o[11] = 0.0; o[12] = 0.0;
    }
    __syncthreads();
  }
}

template <bool BWD>
__global__ void __launch_bounds__(ST, 2) k1d_pe_pass2(const PS p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  Tri* wt = reinterpret_cast<Tri*>(smem_raw + 64);               // [2][SNW]
  double* hsS = reinterpret_cast<double*>(smem_raw + 2048);
  double* rhS = hsS + (PCH + 2);
  double* rinB = rhS + (PCH + 2);       // [2] f / gbar row chunk -> x0 -> output staging
  double* kSB = rinB + 2 * PBUF;        // [2] kappa row chunk -> (backward) dL/dkappa_e staging
  double* uSB = kSB + 2 * PBUF;         // [2] backward: u row chunk with one halo node
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x % p.G, col = blockIdx.x / p.G;
  const ChunkP ck = make_chunk_pe(p, c, tid);
  load_mesh_chunk_pe(p, ck, hsS, rhS, tid);
  for (int j = tid; j < 2 * PBUF; j += ST) kSB[j] = 1.0;
  if (tid == 0) {
    mbar_init_raw(bar, 1);
    mbar_init_raw(bar + 1, 1);
    fence_mbar_init();
  }
  fence_async_smem();
  __syncthreads();
  const double* hsT = hsS + ck.tb;
  const double* rhT = rhS + ck.tb;
  const int ulen = BWD ? ck.len + ((ck.n0 + ck.len < p.nn) ? 1 : 0) : 0;
  const bool shared_field = (p.ldk == 0);
  double gacc[PR];
#pragma unroll
  for (int j = 0; j < PR; ++j) gacc[j] = 0.0;
  auto issue = [&](long long s, int b) {   // thread 0: rows of sample s -> buffer set b
    const double* g0 = p.in0 + s * p.ld0 + ck.n0;
    const double* gk = p.kap_row + s * p.ldk + ck.eA;
    const double* gu = BWD ? p.in1 + s * p.ld1 + ck.n0 : nullptr;
    const bool l0 = s == p.B - 1 && c == p.G - 1;
    const bool lk = (p.ldk == 0 || s == p.B - 1) && ck.eA + ck.ecnt == p.nn - 1;
    const bool lu = s == p.B - 1 && ck.n0 + ulen == p.nn;
    double* rb = rinB + b * PBUF;
    double* kb = kSB + b * PBUF + 2;
    double* ub = uSB + b * PBUF;
    row_scalars(rb, g0, ck.len, p.sup0, l0);
    row_scalars(kb, gk, ck.ecnt, p.supk, lk);
    if (BWD) row_scalars(ub, gu, ulen, p.sup1, lu);
    mbar_arrive_expect_tx(bar + b, row_tx_bytes(g0, ck.len, p.sup0, l0) + row_tx_bytes(gk, ck.ecnt, p.supk, lk) +
                                       (BWD ? row_tx_bytes(gu, ulen, p.sup1, lu) : 0u));
    row_bulk(rb, g0, ck.len, p.sup0, l0, bar + b);
    row_bulk(kb, gk, ck.ecnt, p.supk, lk, bar + b);
    if (BWD) row_bulk(ub, gu, ulen, p.sup1, lu, bar + b);
  };

  int it = 0;
  long long s = p.s_begin + col;
  if (tid == 0 && s < p.s_end) issue(s, 0);
  for (; s < p.s_end; s += p.NG, ++it) {
    const int bsel = it & 1;
    double* rin = rinB + bsel * PBUF;
    double* kS = kSB + bsel * PBUF;
    const double* uS = uSB + bsel * PBUF;
    const double* g0 = p.in0 + s * p.ld0 + ck.n0;
    const double* gk = p.kap_row + s * p.ldk + ck.eA;
    const double* gu = BWD ? p.in1 + s * p.ld1 + ck.n0 : nullptr;
    const double* cf = p.coef + (s * p.G + c) * NP2;
    const double alpha = cf[0], beta = cf[1], alpha1 = cf[2], beta1 = cf[3];
    const int mi = mis_of(g0);
    const bool have_out = (p.out != nullptr);
    double* go = have_out ? p.out + s * p.ldo + ck.n0 : nullptr;
    const int mo = have_out ? mis_of(go) : 0;
    const double* kT = kS + 2 + mis_of(gk) + ck.tb + ck.koff;
    const double* uT = BWD ? uS + mis_of(gu) + ck.tb : nullptr;
    mbar_wait(bar + bsel, (it >> 1) & 1);

    double v[PR], ikv[PR], ge[PR];   // ikv = 2/kappa_e
    Tri t = tri_id();
    {
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < PR; ++j) {
        const double hi = hsT[j + 1];
        const double in = (j < ck.nin) ? rin[mi + ck.tb + j] : 0.0;
        double v0 = BWD ? in : __dadd_rn(__dmul_rn(hp, in), __dmul_rn(hi, in));
        if (j == 0 && ck.ownsL) v0 = 0.0;
        v[j] = v0;
        const double ik = (j < ck.nev) ? 2.0 * __drcp_rn(kT[j + 1]) : 0.0;   // == RN(2 / kappa_e)
        ikv[j] = ik;
        const double w = hi * ik;   // w_e = h_e/kappa_e (hs = h/2)
        t.s += v0;
        t.w = fma(w, t.s, t.w);
        t.x += w;
        hp = hi;
      }
    }
    Tri tot;
    const Tri ex = cta_excl_scan_pe(t, wt, lane, warp, tot);
    // prefetch the next sample into the other buffer set — here, not at the top of the iteration, so that the bulk stores of
    // the previous sample (which read that set) have had half an iteration to drain
    if (tid == 0 && s + p.NG < p.s_end) {
      bulk_wait_read0();
      issue(s + p.NG, bsel ^ 1);
    }
    Tri t1 = tri_id();
    {
      double S = ex.s, X = ex.x, W = ex.w;
      double kp = ck.e0 ? kdiv(0.5 * kT[0], hsT[0], rhT[0]) : 0.0;
#pragma unroll
      for (int j = 0; j < PR; ++j) {
        S += v[j];
        const double x0 = fma(beta, X, alpha) - W;
        if (have_out) rin[mo + ck.tb + j] = x0;
        if (BWD) ge[j] = (j < ck.nev) ? (beta - S) * (uT[j + 1] - uT[j]) : 0.0;   // q0_e (u_{e+1}-u_e)
        const double ki = (j < ck.nev) ? kdiv(0.5 * kT[j + 1], hsT[j + 1], rhT[j + 1]) : 0.0;
        const double v1 = __dmul_rn(two_sum_err(kp, ki), x0);
        kp = ki;
        v[j] = v1;
        const double w = hsT[j + 1] * ikv[j];
        W = fma(w, S, W);
        X += w;
        t1.s += v1;
        t1.w = fma(w, t1.s, t1.w);
        t1.x += w;
      }
    }
    const Tri ex1 = cta_excl_scan_pe(t1, wt + SNW, lane, warp, tot);   // barrier: all kappa reads of this sample done
    {
      double S = ex1.s, X = ex1.x, W = ex1.w;
      double hp = hsT[0];
#pragma unroll
      for (int j = 0; j < PR; ++j) {
        const double hi = hsT[j + 1];
        S += v[j];
        const double x1 = fma(beta1, X, alpha1) - W;
        const double w = hi * ikv[j];
        W = fma(w, S, W);
        X += w;
        if (have_out && j < ck.nst) {
          const double xv = rin[mo + ck.tb + j] + x1;
          rin[mo + ck.tb + j] = BWD ? fma(xv, hp, xv * hi) : xv;
        }
        if (BWD) {
          // dL/dkappa_e = -(q0_e + q1_e)(u_{e+1}-u_e)/kappa_e
          const double du = (j < ck.nev) ? (uT[j + 1] - uT[j]) : 0.0;
          const double g = -(ge[j] + (beta1 - S) * du) * (0.5 * ikv[j]);
          ge[j] = (j < ck.nev) ? g : 0.0;
        }
        hp = hi;
      }
    }
    if (have_out) {
      if (ck.ownsL) rin[mo] = BWD ? 0.0 : p.gL;
      if (ck.ownsR) rin[mo + ck.len - 1] = BWD ? 0.0 : p.gR;
    }
    double* gko = nullptr;
    int mg = 0;
    const int nel_chunk = max(0, min(ck.len, p.nn - 1 - ck.n0));   // elements n0 .. n0+nel_chunk-1 belong to this chunk
    if (BWD) {
      if (shared_field) {
#pragma unroll
        for (int j = 0; j < PR; ++j) gacc[j] += ge[j];   // fixed order over this column's samples
      } else {
        gko = p.gke_out + s * static_cast<long long>(p.nn - 1) + ck.n0;
        mg = mis_of(gko);
#pragma unroll
        for (int j = 0; j < PR; ++j)
          if (j < ck.nev) kS[mg + ck.tb + j] = ge[j];   // kappa chunk no longer needed (barrier above)
      }
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      if (have_out) {
        const Seg qo = make_seg(go, ck.len);
        if (qo.head) go[0] = rin[qo.mis];
        if (qo.tail) go[ck.len - 1] = rin[qo.mis + ck.len - 1];
        if (qo.body) bulk_s2g(go + qo.head, rin + qo.mis + qo.head, 8u * qo.body);
      }
      if (BWD && !shared_field && nel_chunk > 0) {
        const Seg qg = make_seg(gko, nel_chunk);
        if (qg.head) gko[0] = kS[qg.mis];
        if (qg.tail) gko[nel_chunk - 1] = kS[qg.mis + nel_chunk - 1];
        if (qg.body) bulk_s2g(gko + qg.head, kS + qg.mis + qg.head, 8u * qg.body);
      }
      bulk_commit();   // (drained before this buffer set is refilled: see the prefetch above)
    }
  }
  if (BWD && shared_field) {
    double* o = p.gk_cols + static_cast<long long>(col) * (p.nn - 1) + ck.n0 + ck.tb;
#pragma unroll
    for (int j = 0; j < PR; ++j)
      if (j < ck.nev) o[j] = gacc[j];
  }
  if (tid == 0) bulk_wait_read0();
}

// shared per-element field: dL/dkappa_e = sum over CTA columns (fixed order)
__global__ void k1d_gk_cols_sum(const double* cols, int ncols, long long n_el, double* out) {
  const long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if (e >= n_el) return;
  double a = 0.0;
  for (int c = 0; c < ncols; ++c) a += cols[c * n_el + e];
  out[e] = a;
}

// per-sample dL/dkappa -> output (PER_SAMPLE: copy; SCALAR: fixed-order sum over the batch)
__global__ void k1d_gk_out(const double* gk, long long B, int per_sample, double* out) {
  if (per_sample) {
    const long long s = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (s < B) out[s] = gk[s];
  } else {
    __shared__ double sh[1024];
    double a = 0.0;
    for (long long i = threadIdx.x; i < B; i += blockDim.x) a += gk[i];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int d = blockDim.x / 2; d > 0; d >>= 1) {
      if (static_cast<int>(threadIdx.x) < d) sh[threadIdx.x] += sh[threadIdx.x + d];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
  }
}

constexpr size_t smem_p1(bool bwd) { return 2048 + sizeof(double) * (2 * (SCH + 2) + 2 * (SCH + 4)) + (bwd ? 0 : 0); }
constexpr size_t smem_p2() { return 2048 + sizeof(double) * (2 * (SCH + 2) + 2 * (SCH + 4)); }

}  // namespace

namespace dfe {

size_t split1d_workspace_bytes(const dfe_mesh* m, long long B) {
  const int nn = static_cast<int>(m->info.n_nodes);
  const size_t G = static_cast<size_t>((nn + PCH - 1) / PCH);   // the per-element kernels use the smaller chunk
  return static_cast<size_t>(B) * G * (NP1 + NP2) * sizeof(double) + static_cast<size_t>(B) * sizeof(double) +
         (static_cast<size_t>(2 * 160) * PCH + static_cast<size_t>(nn)) * sizeof(double) + 1024;
}

// Runs forward (gbar == nullptr) or backward.  Returns DFE_OK or an error; never falls back.
int split1d_run(const dfe_mesh* m, long long B, bool bwd, const double* in0, long long ld0, const double* in1,
                long long ld1, const double* kappa, int kappa_mode, double* out, long long ldo, double* gkappa,
                void* ws, cudaStream_t st) {
  const bool pe = kappa_mode == DFE_KAPPA_PER_ELEMENT || kappa_mode == DFE_KAPPA_PER_SAMPLE_ELEMENT;
  const int per_sample = kappa_mode == DFE_KAPPA_PER_SAMPLE;
  const int chcap = pe ? PCH : SCH;
  PS p{};
  p.nn = static_cast<int>(m->info.n_nodes);
  p.G = (p.nn + chcap - 1) / chcap;
  p.chg = (p.nn + p.G - 1) / p.G;
  p.B = B;
  p.hs = m->d_hs;
  p.rh = m->d_rh;
  p.in0 = in0; p.ld0 = ld0; p.in1 = in1; p.ld1 = ld1; p.out = out; p.ldo = ldo;
  p.kappa = kappa; p.per_sample = per_sample;
  p.bcL = m->bc_left; p.bcR = m->bc_right; p.gL = m->g_left; p.gR = m->g_right;
  unsigned char* w = static_cast<unsigned char*>(ws);
  p.part = reinterpret_cast<double*>(w);
  p.coef = p.part + static_cast<size_t>(B) * p.G * NP1;
  p.gk = p.coef + static_cast<size_t>(B) * p.G * NP2;
  p.gk_cols = p.gk + B;
  if (pe) {
    p.kap_row = kappa;
    p.ldk = kappa_mode == DFE_KAPPA_PER_SAMPLE_ELEMENT ? p.nn - 1 : 0;
    p.gke_out = gkappa;
    p.gk = nullptr;   // the fold kernel does not produce a scalar gradient in these modes
    p.sup0 = (reinterpret_cast<uintptr_t>(in0) & 15) == 0;
    p.sup1 = in1 && (reinterpret_cast<uintptr_t>(in1) & 15) == 0;
    p.supk = (reinterpret_cast<uintptr_t>(kappa) & 15) == 0;
  }

  {   // per device / context, so set on every call (a process may drive several GPUs); a host-side table update
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pass1<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p1(false)));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pass1<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p1(true)));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pass2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p2()));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pass2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_p2()));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pe_pass1<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pe(2)));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pe_pass1<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pe(2)));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pe_pass2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pe(2)));
    DFE_CUDA_OK(cudaFuncSetAttribute(k1d_pe_pass2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pe(3)));
  }
  // Slabs: the batch is walked in groups of samples whose rows fit the L2, so that pass 2's re-read of
  // the row is an L2 hit.  DFE_1D_SLAB_MB overrides the slab size (0 = whole batch in one slab).
  static const long long slab_mb = [] {
    const char* e = getenv("DFE_1D_SLAB_MB");
    return e ? atoll(e) : 0LL;
  }();
  const long long row_bytes = static_cast<long long>(p.nn) * 8 * (bwd ? 2 : 1);
  long long slab = (slab_mb > 0 && !pe) ? (slab_mb << 20) / row_bytes : B;   // per-element kernels: one slab
  const long long cols_full = (2LL * m->sm_count) / p.G > 0 ? (2LL * m->sm_count) / p.G : 1;   // CTA columns per wave
  if (slab < cols_full) slab = cols_full;
  if (slab > B) slab = B;
  for (long long s0 = 0; s0 < B; s0 += slab) {
    p.s_begin = s0;
    p.s_end = s0 + slab < B ? s0 + slab : B;
    const long long ns = p.s_end - p.s_begin;
    long long NG = cols_full < ns ? cols_full : ns;
    p.NG = static_cast<int>(NG);
    const unsigned grid = static_cast<unsigned>(NG * p.G);
    const unsigned fold_blocks = static_cast<unsigned>((ns * 32 + 127) / 128);
    if (pe) {
      if (NG > 160) NG = 160;   // bound of the per-column partial buffer
      p.NG = static_cast<int>(NG);
      const unsigned gpe = static_cast<unsigned>(NG * p.G);
      if (!bwd) {
        k1d_pe_pass1<false><<<gpe, ST, smem_pe(2), st>>>(p);
        k1d_fold<false><<<fold_blocks, 128, 0, st>>>(p);
        k1d_pe_pass2<false><<<gpe, ST, smem_pe(2), st>>>(p);
      } else {
        k1d_pe_pass1<true><<<gpe, ST, smem_pe(2), st>>>(p);
        k1d_fold<true><<<fold_blocks, 128, 0, st>>>(p);
        k1d_pe_pass2<true><<<gpe, ST, smem_pe(3), st>>>(p);
        if (p.ldk == 0) {
          const long long n_el = p.nn - 1;
          k1d_gk_cols_sum<<<static_cast<unsigned>((n_el + 255) / 256), 256, 0, st>>>(p.gk_cols, p.NG, n_el, gkappa);
        }
      }
    } else if (!bwd) {
      k1d_pass1<false><<<grid, ST, smem_p1(false), st>>>(p);
      k1d_fold<false><<<fold_blocks, 128, 0, st>>>(p);
      k1d_pass2<false><<<grid, ST, smem_p2(), st>>>(p);
    } else {
      k1d_pass1<true><<<grid, ST, smem_p1(true), st>>>(p);
      k1d_fold<true><<<fold_blocks, 128, 0, st>>>(p);
      if (out) k1d_pass2<true><<<grid, ST, smem_p2(), st>>>(p);
    }
  }
  if (bwd && !pe) {
    if (per_sample) k1d_gk_out<<<static_cast<unsigned>((B + 255) / 256), 256, 0, st>>>(p.gk, B, 1, gkappa);
    else k1d_gk_out<<<1, 1024, 0, st>>>(p.gk, B, 0, gkappa);
  }
  DFE_CUDA_OK(cudaGetLastError());
  return DFE_OK;
}

}  // namespace dfe
