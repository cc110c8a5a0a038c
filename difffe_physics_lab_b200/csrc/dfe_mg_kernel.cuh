// The persistent solve kernel of dfe_mg.cu and the level phases it is made of.  Included TWICE by dfe_mg.cu, inside a namespace
// per CTA size (MG_KERNEL_NS / MG_KERNEL_MT): 768 threads per CTA for large grids, 512 for grids of at most 65 536 unknowns
// (measured: config 3 1.06 -> 0.93 ms per solve; config 4 is bound by its grid barriers and does not care).  Everything in here
// is identical for both; only MT / MW differ.
namespace MG_KERNEL_NS {
constexpr int MT = MG_KERNEL_MT;   // threads per CTA, one CTA per SM
constexpr int MW = MT / 32;

// How the phases of a group of levels are separated: by the grid-wide barrier (every CTA works on its range of the
// level) or, for the small levels that CTA 0 handles alone out of its shared memory, by a CTA barrier.
struct GridPhase {
  const GridSync& gs;
  unsigned int& epoch;
  double* sh;
  __device__ __forceinline__ void range(int n, int& lo, int& hi) const { cta_range(n, lo, hi); }
  __device__ __forceinline__ void sync() const { grid_barrier<MW>(gs, epoch, sh); }
  __device__ __forceinline__ void sync_sum(double& v) const {
    double zero = 0.0;
    grid_sum2<MW>(gs, epoch, v, zero, sh);
  }
};
struct CtaPhase {
  __device__ __forceinline__ void range(int n, int& lo, int& hi) const { lo = 0; hi = n; }
  __device__ __forceinline__ void sync() const { __syncthreads(); }
  __device__ __forceinline__ void sync_sum(double&) const { __syncthreads(); }
};

// One level on the way down: pre-smoothing (sweep 1 starts from zero and is never materialised: x1 = omega D^-1 b),
// residual, restriction into bc (the right-hand side of the next level).  Returns the pre-smoothed iterate
// (nullptr: the implicit x1).
template <class Ph>
__device__ __forceinline__ const double* mg_down(const MgMat& M, const MgVec& V, const MgMat& Mc, double* bc, int nu,
                                                 const double* om, const Ph& ph) {
  const int tid = threadIdx.x;
  int lo, hi;
  ph.range(M.n, lo, hi);
  const double* b = V.b;
  const double* dinv = M.dinv;
  const double om1 = om[0];
  auto x1 = [&](int k) { return om1 * dinv[k] * b[k]; };
  const double* src = nullptr;
  for (int s = 2; s <= nu; ++s) {
    double* dst = (src == V.xa) ? V.xb : V.xa;
    const double OMEGA = om[s - 1];
    for (int k = lo + tid; k < hi; k += MT) {
      const int i = k / M.mx, j = k - i * M.mx;
      double xo, off;
      if (src) { xo = src[k]; off = offsum(M, i, j, k, [&](int q) { return src[q]; }); }
      else { xo = x1(k); off = offsum(M, i, j, k, x1); }
      dst[k] = fma(OMEGA * dinv[k], b[k] - off, (1.0 - OMEGA) * xo);
    }
    ph.sync();
    src = dst;
  }
  for (int k = lo + tid; k < hi; k += MT) {   // r = b - A x
    const int i = k / M.mx, j = k - i * M.mx;
    double xo, off;
    if (src) { xo = src[k]; off = offsum(M, i, j, k, [&](int q) { return src[q]; }); }
    else { xo = x1(k); off = offsum(M, i, j, k, x1); }
    V.r[k] = b[k] - fma(M.C[k], xo, off);
  }
  ph.sync();
  int clo, chi;
  ph.range(Mc.n, clo, chi);
  for (int k = clo + tid; k < chi; k += MT) {   // b_{l+1} = P^T r
    const int I = k / Mc.mx, J = k - I * Mc.mx;
    const int fi = 2 * I + 1, fj = 2 * J + 1;
    double sum = 0.0;
#pragma unroll
    for (int di = -1; di <= 1; ++di)
#pragma unroll
      for (int dj = -1; dj <= 1; ++dj) {
        const int pi = fi + di, pj = fj + dj;
        if (pi < 0 || pi >= M.my || pj < 0 || pj >= M.mx) continue;
        sum = fma(pweight(M, pi, pj, I, J), V.r[pi * M.mx + pj], sum);
      }
    bc[k] = sum;
  }
  ph.sync();
  return src;
}

// One level on the way up: y = x + P e, then nu post-smoothing sweeps.  `rz` (finest level only): the last sweep also
// forms sum_k b_k x_k and the closing barrier reduces it over the grid.  Returns the final iterate.
template <class Ph>
__device__ __forceinline__ const double* mg_up(const MgMat& M, const MgVec& V, const double* src, const double* e,
                                               int nu, const double* om, double* rz, const Ph& ph) {
  const int tid = threadIdx.x;
  int lo, hi;
  ph.range(M.n, lo, hi);
  const double* b = V.b;
  const double* dinv = M.dinv;
  const int cy = M.my >> 1, cx = M.mx >> 1;
  const size_t n = M.n;
  double* dst = (src == V.xa) ? V.xb : V.xa;
  for (int k = lo + tid; k < hi; k += MT) {
    const int i = k / M.mx, j = k - i * M.mx;
    const bool oi = i & 1, oj = j & 1;
    double c;
    if (oi && oj) {
      c = e[(i >> 1) * cx + (j >> 1)];
    } else if (oi) {
      const int I = i >> 1, JE = j >> 1, JW = JE - 1;
      c = (JW >= 0 ? M.pw[k] * e[I * cx + JW] : 0.0) + (JE < cx ? M.pw[n + k] * e[I * cx + JE] : 0.0);
    } else if (oj) {
      const int J = j >> 1, IN = i >> 1, IS = IN - 1;
      c = (IS >= 0 ? M.pw[k] * e[IS * cx + J] : 0.0) + (IN < cy ? M.pw[n + k] * e[IN * cx + J] : 0.0);
    } else {
      const int IN = i >> 1, IS = IN - 1, JE = j >> 1, JW = JE - 1;
      c = 0.0;
      if (IS >= 0 && JW >= 0) c = fma(M.pw[k], e[IS * cx + JW], c);
      if (IS >= 0 && JE < cx) c = fma(M.pw[n + k], e[IS * cx + JE], c);
      if (IN < cy && JW >= 0) c = fma(M.pw[2 * n + k], e[IN * cx + JW], c);
      if (IN < cy && JE < cx) c = fma(M.pw[3 * n + k], e[IN * cx + JE], c);
    }
    dst[k] = (src ? src[k] : om[0] * dinv[k] * b[k]) + c;
  }
  ph.sync();
  src = dst;
  for (int s = 1; s <= nu; ++s) {
    dst = (src == V.xa) ? V.xb : V.xa;
    const bool last = (rz != nullptr && s == nu);
    const double OMEGA = om[nu - s];   // the pre-smoother's weights in reverse order: the cycle stays symmetric
    double acc = 0.0;
    for (int k = lo + tid; k < hi; k += MT) {
      const int i = k / M.mx, j = k - i * M.mx;
      const double off = offsum(M, i, j, k, [&](int q) { return src[q]; });
      const double xn = fma(OMEGA * dinv[k], b[k] - off, (1.0 - OMEGA) * src[k]);
      dst[k] = xn;
      if (last) acc = fma(b[k], xn, acc);
    }
    if (last) {
      ph.sync_sum(acc);
      *rz = acc;
    } else {
      ph.sync();
    }
    src = dst;
  }
  return src;
}


__global__ void __launch_bounds__(MT, 1) k_mgpcg(const __grid_constant__ MgArgs A) {
  extern __shared__ __align__(16) double tail_smem[];
  __shared__ double sh[2 * MW + 2];
  unsigned int epoch = 0;
  const GridSync gs{A.slots, A.abort_flag, A.backoff};
  const GridPhase gph{gs, epoch, sh};
  const CtaPhase cph{};
  const int tid = threadIdx.x;
  const int L = A.H.L, nu = A.nu;
  const MgMat& F = A.H.lev[0];
  double* const rcg = A.v[0].b;       // the CG residual is the right-hand side of the finest level
  int lo0, hi0;
  cta_range(F.n, lo0, hi0);

  // ---- the tail of the hierarchy: first level lc with n <= TAIL_N (lc >= 1).  CTA 0 keeps copies of those levels'
  // matrices and work vectors in shared memory; b / xa / xb of level lc itself stay in global memory (they are the
  // interface to the other CTAs).
  int lc = L - 1;
  while (lc > 1 && A.H.lev[lc - 1].n <= TAIL_N) --lc;
  MgMat tm[MG_MAXL];
  MgVec tv[MG_MAXL];
  if (blockIdx.x == 0) {
    double* sp = tail_smem;
    for (int l = lc; l < L; ++l) {
      const MgMat& G = A.H.lev[l];
      MgMat& T = tm[l];
      T = G;
      const size_t n = G.n;
      T.C = sp; sp += n;
      T.dinv = sp; sp += n;
      T.E = sp; sp += n;
      T.N = sp; sp += n;
      T.NE = sp; sp += n;
      T.NW = sp; sp += n;
      for (int k = tid; k < G.n; k += MT) {
        T.C[k] = G.C[k]; T.dinv[k] = G.dinv[k]; T.E[k] = G.E[k]; T.N[k] = G.N[k];
        T.NE[k] = G.nine ? G.NE[k] : 0.0;
        T.NW[k] = G.nine ? G.NW[k] : 0.0;
      }
      T.nine = 1;
      if (l + 1 < L) {
        T.pw = sp; sp += 4 * n;
        for (int k = tid; k < 4 * G.n; k += MT) T.pw[k] = G.pw[k];
      }
      tv[l].r = sp; sp += n;
      if (l == lc) {
        tv[l].b = A.v[l].b; tv[l].xa = A.v[l].xa; tv[l].xb = A.v[l].xb;
      } else {
        tv[l].b = sp; sp += n;
        tv[l].xa = sp; sp += n;
        tv[l].xb = sp; sp += n;
      }
    }
    __syncthreads();
  }

  // ---- init: x = 0, p buffers = 0, amax = max |rhs_k|
  double amax = 0.0;
  for (int k = lo0 + tid; k < hi0; k += MT) {
    amax = fmax(amax, fabs(A.rhs[k]));
    A.x[k] = 0.0;
    A.p0[k] = 0.0;
    A.p1[k] = 0.0;
  }
  amax = grid_max<MW>(gs, epoch, amax, sh);
  // Solve for 2^sc rhs with max |2^sc rhs_k| in [1, 2), as k_pcg does: no square underflows or overflows, and since the
  // V-cycle is linear too (smoothing, restriction, prolongation, the coarsest inverse), in-range inputs keep their bits.
  int sc = 0;
  if (amax > 0.0 && isfinite(amax)) {
    frexp(amax, &sc);
    sc = 1 - sc;
  }
  // ---- r = 2^sc rhs
  double bb = 0.0, zero = 0.0;
  for (int k = lo0 + tid; k < hi0; k += MT) {
    const double bi = ldexp(A.rhs[k], sc);
    rcg[k] = bi;
    bb = fma(bi, bi, bb);
  }
  grid_sum2<MW>(gs, epoch, bb, zero, sh);
  const double bnorm = sqrt(bb);
  double status = 0.0, relres = 0.0;
  long long it = 0;
  // a non-finite rhs: amax = inf gives bb = inf (or NaN); fmax drops a NaN, but the sum does not
  if (!isfinite(bb)) {
    status = 5.0;
  } else if (bb == 0.0) {
    // rhs == 0 -> x = 0
  } else {
    double rz = 0.0, beta = 0.0;
    double* pold = A.p0;
    double* pnew = A.p1;
    status = 4.0;
    while (it < A.maxit) {
      // ======================================================= z = M^{-1} r : one V(nu, nu) cycle
      const double* xsrc[MG_MAXL];    // pre-smoothed iterate of every level (nullptr: the implicit first sweep)
      double rz_new = 0.0;
      for (int l = 0; l < lc; ++l) xsrc[l] = mg_down(A.H.lev[l], A.v[l], A.H.lev[l + 1], A.v[l + 1].b, nu, A.omega, gph);
      if (blockIdx.x == 0) {          // the tail: levels lc .. L-1, CTA 0 alone
        for (int l = lc; l + 1 < L; ++l) xsrc[l] = mg_down(tm[l], tv[l], tm[l + 1], tv[l + 1].b, nu, A.omega, cph);
        const int nc = A.H.nc;
        if (tid < nc) {               // coarsest level: x = Ainv b
          const double* b = tv[L - 1].b;
          double sum = 0.0;
          for (int c = 0; c < nc; ++c) sum = fma(A.H.cinv[tid * nc + c], b[c], sum);
          tv[L - 1].xa[tid] = sum;
        }
        __syncthreads();
        const double* e = tv[L - 1].xa;
        for (int l = L - 2; l >= lc; --l) e = mg_up(tm[l], tv[l], xsrc[l], e, nu, A.omega, nullptr, cph);
        // (for lc == L-1 the coarsest solution itself sits in the global xa of that level)
      }
      grid_barrier<MW>(gs, epoch, sh);
      // which buffer of level lc holds its final iterate is a function of nu alone (every CTA can tell)
      const double* e;
      if (lc == L - 1) {
        e = A.v[lc].xa;
      } else {
        // mg_down leaves the iterate in xa after an even number of explicit sweeps (nu - 1 of them), mg_up adds 1 + nu writes
        const double* src = (nu >= 2) ? (((nu - 1) & 1) ? A.v[lc].xa : A.v[lc].xb) : nullptr;
        const double* cur = (src == A.v[lc].xa) ? A.v[lc].xb : A.v[lc].xa;   // after y = x + P e
        for (int s = 1; s <= nu; ++s) cur = (cur == A.v[lc].xa) ? A.v[lc].xb : A.v[lc].xa;
        e = cur;
      }
      for (int l = lc - 1; l >= 0; --l) e = mg_up(A.H.lev[l], A.v[l], xsrc[l], e, nu, A.omega, l == 0 ? &rz_new : nullptr, gph);
      if (grid_aborted(gs)) { status = 7.0; break; }
      const double* z = e;
      if (!(rz_new > 0.0) || !isfinite(rz_new)) { status = 5.0; break; }
      beta = it > 0 ? rz_new / rz : 0.0;
      rz = rz_new;
      // ======================================================= CG phase A: p = z + beta p_old, q = A p, p . q
      double pq = 0.0;
      for (int k = lo0 + tid; k < hi0; k += MT) {
        const int i = k / F.mx, j = k - i * F.mx;
        auto pv = [&](int q) { return fma(beta, pold[q], z[q]); };
        const double pk = pv(k);
        const double qk = fma(F.C[k], pk, offsum(F, i, j, k, pv));
        pnew[k] = pk;
        A.q[k] = qk;
        pq = fma(pk, qk, pq);
      }
      grid_sum2<MW>(gs, epoch, pq, zero, sh);
      if (grid_aborted(gs)) { status = 7.0; break; }
      if (!(pq > 0.0) || !isfinite(pq)) { status = 5.0; break; }
      const double alpha = rz / pq;
      // ======================================================= CG phase B: x += alpha p, r -= alpha q, r . r
      double rr = 0.0;
      for (int k = lo0 + tid; k < hi0; k += MT) {
        A.x[k] = fma(alpha, pnew[k], A.x[k]);
        const double rk = fma(-alpha, A.q[k], rcg[k]);
        rcg[k] = rk;
        rr = fma(rk, rk, rr);
      }
      grid_sum2<MW>(gs, epoch, rr, zero, sh);
      if (grid_aborted(gs)) { status = 7.0; break; }
      ++it;
      relres = sqrt(rr) / bnorm;
      if (!isfinite(rr)) { status = 5.0; break; }
      if (sqrt(rr) <= A.tol * bnorm) { status = 0.0; break; }
      double* t = pold;
      pold = pnew;
      pnew = t;
    }
  }
  // ---- x = 2^-sc x on this CTA's range of level 0 (the threads that last wrote it; nothing reads x after this)
  for (int k = lo0 + tid; k < hi0; k += MT) A.x[k] = ldexp(A.x[k], -sc);
  if (blockIdx.x == 0 && tid == 0) {
    A.out[0] = static_cast<double>(it);
    A.out[1] = relres;
    A.out[2] = status;
    A.out[3] = isfinite(bnorm) ? 0.0 : 1.0;
  }
}

}  // namespace MG_KERNEL_NS
