// Jacobi-preconditioned conjugate gradients on the SELL-32 copy of K_free, one cooperative
// persistent kernel per solve (sm_100a).
//
// Replaces torch.linalg.solve(K_free, F_free) (diffhe/solver.py:174) and — called with gbar_free —
// the adjoint solve inside LinalgSolveExBackward0 (K_free is symmetric, SURVEY §8a row A7).
//
// Layout: warp w owns SELL slices w, w+W, ...; lane l owns row 32*slice+l, so every load of
// sell_val / sell_col is a fully coalesced 256 B / 128 B request.  Per iteration two phases, each
// ended by one grid-wide barrier (hand-rolled: release-increment + acquire-poll, see grid_barrier):
//   A  p = z + beta p_old (recomputed on the fly for the gathered neighbours, ping-pong p buffers)
//      q = K p ;  partial p.q
//   B  x += alpha p ; r -= alpha q ; z = D^{-1} r ; partial r.z and r.r
// Dot products are reduced in a fixed order (lane-strided sum + xor-shuffle tree over the per-CTA
// partials), identically on every CTA: results are bit-reproducible and no float atomics are used.
// Stops when the recursive residual satisfies ||r||_2 <= tol ||rhs||_2.  The solve runs on 2^sc rhs, the power of two that
// brings max |rhs_i| into [1, 2), and scales x back at the end: exact, and no square underflows or overflows.
#include <cstdlib>

#include "dfe_internal.h"

namespace {

#include "dfe_gridsync.cuh"   // grid_sum2: fixed-order grid reduction fused with the phase barrier, bounded polls

constexpr int PT = 768;  // threads per CTA: one CTA per SM (148 arrivals per grid barrier instead of 444)
constexpr int PW = PT / 32;

struct PcgArgs {
  int n, n_slices;
  const int* slice_ptr;
  const int* col;
  const double* val;
  const double* dinv;
  const double* b;
  double* x;
  double* r;
  double* z;
  double* p0;
  double* p1;
  double* q;
  double* part;   // [3 epochs][gridDim.x][2] exchange slots, pre-set to the sentinel
  double* out;    // [0]=iterations, [1]=relres, [2]=status (0 ok, 4 not converged, 5 breakdown, 7 barrier timeout),
                  // [3]=1 if the breakdown is a non-finite rhs
  int* abort_flag; // zeroed before the launch; raised by a grid barrier that waited longer than its bound
  double tol;
  long long maxit;
  int backoff;    // cycles an early arriver waits between two polls of a slot
};

__global__ void __launch_bounds__(PT, 1) k_pcg(const PcgArgs A) {
  unsigned int epoch = 0;
  __shared__ double sh[2 * PW + 2];
  const GridSync gs{A.part, A.abort_flag, A.backoff};
  const int lane = threadIdx.x & 31;
  // A CTA owns a CONTIGUOUS block of SELL slices and walks it front to back, PW slices at a time: the neighbours a
  // row gathers (rows +-1 and, on a structured mesh, +- one mesh line) were touched by this SM a trip or two ago and
  // are served by its L1 instead of travelling from L2 to two or three different SMs.
  const int per_cta = (A.n_slices + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int s_lo = blockIdx.x * per_cta;
  const int s_hi = s_lo + per_cta < A.n_slices ? s_lo + per_cta : A.n_slices;
  const int gw = s_lo + (threadIdx.x >> 5);
  constexpr int nwarps = PW;

  // ---- init: x = 0, p buffers = 0, amax = max |b_i|
  double amax = 0.0;
  for (int s = gw; s < s_hi; s += nwarps) {
    const int i = 32 * s + lane;
    if (i < A.n) {
      amax = fmax(amax, fabs(A.b[i]));
      A.x[i] = 0.0;
      A.p0[i] = 0.0;
      A.p1[i] = 0.0;
    }
  }
  amax = grid_max<PW>(gs, epoch, amax, sh);
  // Solve for 2^sc b with max |2^sc b_i| in [1, 2): ||b||^2, tol ||b|| and p.q then neither underflow (|b| < ~1e-162 gave
  // bb == 0, i.e. "converged" at x = 0; below ~1e-154 the loop stopped far above tol) nor overflow (|b| ~ 1e155 overflowed
  // p.q into a breakdown).  Where no intermediate leaves the normal range the iterates are those of the unscaled solve,
  // scaled, so relres, the iteration count and (after the scale back below) x keep their bits.
  int sc = 0;
  if (amax > 0.0 && isfinite(amax)) {    // (0: nothing to solve; inf: reported as a breakdown below)
    frexp(amax, &sc);
    sc = 1 - sc;
  }
  // ---- r = 2^sc b, z = D^{-1} r
  double bb = 0.0, rz = 0.0;
  for (int s = gw; s < s_hi; s += nwarps) {
    const int i = 32 * s + lane;
    if (i < A.n) {
      const double bi = ldexp(A.b[i], sc);
      const double zi = A.dinv[i] * bi;
      A.r[i] = bi;
      A.z[i] = zi;
      bb = fma(bi, bi, bb);
      rz = fma(bi, zi, rz);
    }
  }
  grid_sum2<PW>(gs, epoch, bb, rz, sh);
  const double bnorm = sqrt(bb);
  double status = 0.0, relres = 0.0;
  long long it = 0;
  // a non-finite rhs: amax = inf gives bb = inf (or NaN); fmax drops a NaN, but the sum does not
  if (!isfinite(bb)) {
    status = 5.0;
  } else if (bb == 0.0) {
    // rhs == 0 -> x = 0
  } else {
    double beta = 0.0;
    double* pold = A.p0;
    double* pnew = A.p1;
    status = 4.0;
    while (it < A.maxit) {
      // ---- phase A
      double pq = 0.0;
      for (int s = gw; s < s_hi; s += 2 * nwarps) {
        // two slices per trip, four columns of each per batch: all column / value loads of a batch are issued
        // before the first dependent gather, so ~16 gathers per thread are in flight (the kernel is bound by
        // memory latency, not bandwidth: ncu long_scoreboard 73 % with one column at a time)
        const int s2 = s + nwarps;
        const bool has2 = s2 < s_hi;
        const int i = 32 * s + lane, i2 = 32 * s2 + lane;
        const int beg = A.slice_ptr[s], end = A.slice_ptr[s + 1];
        const int beg2 = has2 ? A.slice_ptr[s2] : 0, end2 = has2 ? A.slice_ptr[s2 + 1] : 0;
        const int wd = (end - beg) >> 5, wd2 = (end2 - beg2) >> 5;
        const int wmax = wd > wd2 ? wd : wd2;
        double sum = 0.0, sum2 = 0.0;
        for (int w0 = 0; w0 < wmax; w0 += 4) {
          int j[4], j2[4];
          double v[4], v2[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const bool on = w0 + u < wd, on2 = w0 + u < wd2;
            const int k = beg + ((w0 + u) << 5) + lane, k2 = beg2 + ((w0 + u) << 5) + lane;
            // the matrix streams through once per iteration (evict-first), the vectors it is applied to stay in L2
            j[u] = on ? __ldcs(A.col + k) : -1;
            v[u] = on ? __ldcs(A.val + k) : 0.0;
            j2[u] = on2 ? __ldcs(A.col + k2) : -1;
            v2[u] = on2 ? __ldcs(A.val + k2) : 0.0;
          }
          double g[4], g2[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            g[u] = j[u] >= 0 ? fma(beta, pold[j[u]], A.z[j[u]]) : 0.0;
            g2[u] = j2[u] >= 0 ? fma(beta, pold[j2[u]], A.z[j2[u]]) : 0.0;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {   // same accumulation order as a column-by-column loop
            if (j[u] >= 0) sum = fma(v[u], g[u], sum);
            if (j2[u] >= 0) sum2 = fma(v2[u], g2[u], sum2);
          }
        }
        if (i < A.n) {
          const double pi = fma(beta, pold[i], A.z[i]);
          pnew[i] = pi;
          A.q[i] = sum;
          pq = fma(pi, sum, pq);
        }
        if (has2 && i2 < A.n) {
          const double pi = fma(beta, pold[i2], A.z[i2]);
          pnew[i2] = pi;
          A.q[i2] = sum2;
          pq = fma(pi, sum2, pq);
        }
      }
      double unused = 0.0;
      grid_sum2<PW>(gs, epoch, pq, unused, sh);
      if (grid_aborted(gs)) {
        status = 7.0;
        break;
      }
      if (!(pq > 0.0) || !isfinite(pq)) {
        status = 5.0;
        break;
      }
      const double alpha = rz / pq;
      // ---- phase B
      double rz_new = 0.0, rr = 0.0;
      for (int s = gw; s < s_hi; s += 2 * nwarps) {   // two slices per trip: ten independent loads in flight
        const int i = 32 * s + lane, i2 = i + 32 * nwarps;
        const bool on = i < A.n, on2 = (s + nwarps < s_hi) && i2 < A.n;
        double xi = 0, pi = 0, qi = 0, ri = 0, di = 0, xi2 = 0, pi2 = 0, qi2 = 0, ri2 = 0, di2 = 0;
        // x is touched once per iteration and never gathered: streamed (evict-first) like the matrix
        if (on) { xi = __ldcs(A.x + i); pi = pnew[i]; qi = A.q[i]; ri = A.r[i]; di = A.dinv[i]; }
        if (on2) { xi2 = __ldcs(A.x + i2); pi2 = pnew[i2]; qi2 = A.q[i2]; ri2 = A.r[i2]; di2 = A.dinv[i2]; }
        if (on) {
          __stcs(A.x + i, fma(alpha, pi, xi));
          ri = fma(-alpha, qi, ri);
          const double zi = di * ri;
          A.r[i] = ri;
          A.z[i] = zi;
          rz_new = fma(ri, zi, rz_new);
          rr = fma(ri, ri, rr);
        }
        if (on2) {
          __stcs(A.x + i2, fma(alpha, pi2, xi2));
          ri2 = fma(-alpha, qi2, ri2);
          const double zi2 = di2 * ri2;
          A.r[i2] = ri2;
          A.z[i2] = zi2;
          rz_new = fma(ri2, zi2, rz_new);
          rr = fma(ri2, ri2, rr);
        }
      }
      grid_sum2<PW>(gs, epoch, rz_new, rr, sh);   // two independent reductions share one exchange
      if (grid_aborted(gs)) {
        status = 7.0;
        break;
      }
      ++it;
      relres = sqrt(rr) / bnorm;
      if (!isfinite(rr)) {
        status = 5.0;
        break;
      }
      if (sqrt(rr) <= A.tol * bnorm) {
        status = 0.0;
        break;
      }
      beta = rz_new / rz;
      rz = rz_new;
      double* t = pold;
      pold = pnew;
      pnew = t;
    }
  }
  // ---- x = 2^-sc x on the rows of this CTA (the threads that last wrote them; nothing reads x after this)
  for (int s = gw; s < s_hi; s += nwarps) {
    const int i = 32 * s + lane;
    if (i < A.n) __stcs(A.x + i, ldexp(__ldcs(A.x + i), -sc));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    A.out[0] = static_cast<double>(it);
    A.out[1] = relres;
    A.out[2] = status;
    A.out[3] = isfinite(bnorm) ? 0.0 : 1.0;
  }
}

struct PcgPlan {
  int grid;
  size_t off_r, off_z, off_p0, off_p1, off_q, off_part, off_out, off_bar, total;
};

int plan_pcg(const dfe_mesh* m, PcgPlan* pl, bool query_device) {
  const size_t n = static_cast<size_t>(m->info.n_free);
  const size_t vec = ((n * sizeof(double) + 255) / 256) * 256;
  int max_grid = 148 * 8;  // upper bound used for workspace sizing
  pl->grid = max_grid;
  if (query_device) {
    int per_sm = 0;
    DFE_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg, PT, 0));
    long long resident = static_cast<long long>(per_sm) * m->sm_count;
    long long want = (static_cast<long long>(m->dev.n_slices) + PW - 1) / PW;  // one slice per warp
    long long g = want < resident ? want : resident;
    if (g < 1) g = 1;
    if (g > max_grid) g = max_grid;
    pl->grid = static_cast<int>(g);
  }
  size_t off = 0;
  pl->off_r = off; off += vec;
  pl->off_z = off; off += vec;
  pl->off_p0 = off; off += vec;
  pl->off_p1 = off; off += vec;
  pl->off_q = off; off += vec;
  pl->off_part = off; off += 6 * static_cast<size_t>(max_grid) * sizeof(double);
  pl->off_out = off; off += 256;
  pl->off_bar = off; off += 256;   // abort word of the bounded grid barriers
  pl->total = off;
  return DFE_OK;
}

}  // namespace

extern "C" size_t dfe_pcg_workspace_bytes(const dfe_mesh* m) {
  if (!m) return 0;
  PcgPlan pl;
  plan_pcg(m, &pl, false);
  return pl.total;
}

extern "C" int dfe_pcg(const dfe_mesh* m, const double* sell_vals, const double* dinv, const double* rhs,
                       double* x, double tol, int64_t maxit, int64_t* iters_host, double* relres_host, void* ws,
                       size_t ws_bytes, void* stream) {
  DFE_REQUIRE(m, "dfe_pcg: mesh is null");
  if (m->info.device < 0) {
    dfe::set_error("dfe_pcg: mesh handle is host-only; no CUDA device (this library has no CPU path)");
    return DFE_ERR_CUDA;
  }
  DFE_REQUIRE(sell_vals && dinv && rhs && x && ws, "dfe_pcg: null argument");
  DFE_REQUIRE(tol > 0.0 && maxit >= 1, "dfe_pcg: tol must be > 0 and maxit >= 1");
  if (iters_host) *iters_host = 0;
  if (relres_host) *relres_host = 0.0;
  if (m->info.n_free == 0) return DFE_OK;
  int prev = -1;
  DFE_CUDA_OK(cudaGetDevice(&prev));
  if (prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  PcgPlan pl;
  int rc = plan_pcg(m, &pl, true);
  if (rc == DFE_OK && ws_bytes < pl.total) {
    dfe::set_error("dfe_pcg: workspace %zu bytes < required %zu", ws_bytes, pl.total);
    rc = DFE_ERR_WORKSPACE;
  }
  if (rc == DFE_OK) {
    unsigned char* w = static_cast<unsigned char*>(ws);
    PcgArgs A{};
    A.n = m->dev.n_free;
    A.n_slices = m->dev.n_slices;
    A.slice_ptr = m->dev.slice_ptr;
    A.col = m->dev.sell_col;
    A.val = sell_vals;
    A.dinv = dinv;
    A.b = rhs;
    A.x = x;
    A.r = reinterpret_cast<double*>(w + pl.off_r);
    A.z = reinterpret_cast<double*>(w + pl.off_z);
    A.p0 = reinterpret_cast<double*>(w + pl.off_p0);
    A.p1 = reinterpret_cast<double*>(w + pl.off_p1);
    A.q = reinterpret_cast<double*>(w + pl.off_q);
    A.part = reinterpret_cast<double*>(w + pl.off_part);
    A.out = reinterpret_cast<double*>(w + pl.off_out);
    A.abort_flag = reinterpret_cast<int*>(w + pl.off_bar);
    A.tol = tol;
    A.maxit = maxit;
    static const int backoff = [] { const char* e = getenv("DFE_PCG_BACKOFF"); return e ? atoi(e) : 250; }();
    A.backoff = backoff;
    void* args[] = {&A};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemsetAsync(A.part, 0xFF, 6 * static_cast<size_t>(pl.grid) * sizeof(double), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(A.abort_flag, 0, sizeof(int), st);
    if (e == cudaSuccess) e = cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_pcg), dim3(pl.grid), dim3(PT), args, 0, st);
    if (e != cudaSuccess) {
      dfe::set_error("dfe_pcg: cooperative launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    } else {
      double out[4] = {0, 0, 0, 0};
      e = cudaMemcpyAsync(out, A.out, sizeof out, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e != cudaSuccess) {
        dfe::set_error("dfe_pcg: %s", cudaGetErrorString(e));
        rc = DFE_ERR_CUDA;
      } else {
        if (iters_host) *iters_host = static_cast<int64_t>(out[0]);
        if (relres_host) *relres_host = out[1];
        if (out[2] == 4.0) {
          dfe::set_error("dfe_pcg: not converged after %lld iterations (relative residual %.3e, tol %.3e)",
                         static_cast<long long>(out[0]), out[1], tol);
          rc = DFE_ERR_NOT_CONVERGED;
        } else if (out[2] == 7.0) {
          dfe::set_error("dfe_pcg: a grid barrier waited longer than its bound (lost co-resident CTA?) at iteration %lld",
                         static_cast<long long>(out[0]));
          rc = DFE_ERR_CUDA;
        } else if (out[2] == 5.0 && out[3] != 0.0) {
          dfe::set_error("dfe_pcg: breakdown at iteration 0: the right-hand side has a non-finite entry (inf or NaN)");
          rc = DFE_ERR_BREAKDOWN;
        } else if (out[2] == 5.0) {
          dfe::set_error("dfe_pcg: breakdown at iteration %lld (p^T K p <= 0 or non-finite): K_free is not SPD — "
                         "does the mesh have a Dirichlet node?",
                         static_cast<long long>(out[0]));
          rc = DFE_ERR_BREAKDOWN;
        }
      }
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}
