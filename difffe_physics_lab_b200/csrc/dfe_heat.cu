// Differentiable heat-equation rollouts: backward Euler with the lumped mass on the banded factor of dfe_band_factor,
//
//   forward   A_ff x_{n+1} = m * x_n + c                                   n = 0 .. N-1
//   adjoint   A_ff lambda_N = gbar_N ;   A_ff lambda_n = gbar_n + m * lambda_{n+1}    n = N-1 .. 1
//
// with A = M_L + dt K(kappa), m = M_L[free], c = dt F_free - (A g)_free, and the gradients
//
//   dL/du0[free] = m * lambda_1 ,   dL/dkappa_e = -dt sum_n sum_b lam~_{n,b}^T K0_e u_{n,b}
//
// (lam~ = lambda scattered with zeros on the Dirichlet nodes, u_n the full state: the kappa-dependence of the lifting is
// included because lam~ vanishes on the Dirichlet rows).  dL/df is W^T (dt sum_n sum_b lam~_n): dfe_grad's gf.
//
// k_heat_roll   the whole time loop in ONE launch.  It runs the block-row step of k_band_solve_mma (dfe_band_mma.cuh) with
//               a time loop around the substitution loop: a warp owns 16 samples for the whole rollout and every lane reads
//               back exactly the row positions it wrote, so consecutive time steps need no synchronisation beyond the
//               per-block-row stage barrier.  The right-hand side is formed at load time (fma(m, x_n, c) forward,
//               fma(m, lambda_{n+1}, gbar_n) adjoint) and the first block of the next step straight from the registers of
//               the last block of this one.  Forward: x_{n+1} is scattered into the node-layout trajectory row with its
//               Dirichlet values.  Adjoint: lambda_n goes to a (N_seg, B, npad) buffer for the gradient kernel and into the
//               running sum sum_n lambda_n (the lane that owns a position updates it: a fixed order).
// k_heat_grad   dL/dkappa_e over all (n, b) pairs of a segment: one CTA per (sample chunk, step) keeps the per-element sums
//               in shared memory while the u rows (node layout) and lambda rows (free layout) stream through a cp.async
//               ring; its partial row goes to (step, chunk) of a (N, n_chunk, n_el) buffer.  The chunking depends on B only,
//               so the sums do not depend on how a rollout was split into checkpoint segments.
// k_heat_gsum   adds the partial rows in a fixed (step, chunk) order and scales by -dt; k_heat_sum1 sums the elements (scalar
//               kappa) in a fixed order.
//
// float64 throughout, no float atomics, every wait bounded.
//
// Per-sample conductivity (kappa (B, 1) or (B, n_el)): one A_b = M_L + dt K(kappa_b) and one factor per sample, so the
// shared B operand of the tensor-core TRSM does not exist; the same recursions run with one warp per sample instead.
// k_hps_shift   A_b = fl(dt K_b), then + M_L on the diagonal: the operations and order of timestepping._HeatOperator, so
//               each A_b is bit-identical to its A (K_b from k_bps_assemble, the factor from k_bps_factor: dfe_band_ps.cu)
// k_hps_cfree   c_b = fl(dt F_free) - (A_b g)_free, the lifting added in the mesh's fixed dict order (lift_ptr / lift_src)
// k_hps_roll    the whole time loop (or one checkpoint segment) in ONE launch, one warp per sample: both sweeps of
//               bps_sweeps per step with the right-hand side formed at load time (fma(m, x_n, c_b) forward,
//               fma(m, lambda_{n+1}, gbar_n[free]) adjoint).  Warps never communicate: no barrier, no wait, no fault word.
// k_hps_grad    gacc (B, n_el) += lam~^T K0_e u, one step at a time in DESCENDING step order (the order the adjoint
//               produces them, within and across checkpoint segments): bit-identical with and without checkpointing, and
//               independent of B.  k_hps_gsum scales by -dt (per element) or sums each sample's elements in a fixed order.
#include "dfe_internal.h"

namespace {

using dfe::MeshDev;
#include "dfe_1d_common.cuh"   // mbarrier / 1-D TMA bulk copy wrappers
#include "dfe_band_mma.cuh"     // block-row step of the tensor-core band solve and its fragment layout
#include "dfe_band_ps_solve.cuh"  // bps_sweeps: both banded sweeps of one sample's factor by one warp

constexpr double AREA_EPS = 1e-15;          // solver.py:120
constexpr long long WAIT_POLLS = 1LL << 24; // try_wait polls before a fragment stage counts as lost (raises the fault word)
constexpr int GT = 256;                     // threads of the gradient kernel
constexpr int GNST = 3;                     // cp.async ring stages of the gradient kernel
constexpr size_t GSMEM_MAX = 200 * 1024;    // shared memory bound of the gradient kernel: sets the mesh size limit
constexpr int GCHUNKS = 64;                 // sample chunks per step of the gradient kernel (fewer for B < 1024)

struct RollArgs {
  int npad, nfree, n_dir, nt;       // nt: time steps of this launch
  long long B;
  const double* Ff;
  const double* Bf;
  const int* fnode;
  const int* dir_idx;
  const double* dir_val;
  const double* mf;                 // (npad) lumped mass on the free rows, zero-padded
  const double* cf;                 // forward: (npad) dt F_free - (A g)_free, zero-padded
  double* X;                        // (B, npad) carry: x_n (forward) / lambda_{n+1} (adjoint); y between the two passes
  const double* u0;                 // forward: (B, .) node-layout initial states, or null: X already holds x_0
  long long ldu0;
  double* traj;                     // forward: state after local step j at traj + b * ld_b + j * ld_t (node layout)
  long long ld_b, ld_t;
  const double* gbar;               // adjoint: dL/du_n at gbar + b * ldg_b + (n / gev - 1) * ldg_t when n % gev == 0
  long long ldg_b, ldg_t;
  int gev, n0;                      // adjoint: steps n0 + nt down to n0 + 1
  double* lam;                      // adjoint: (nt, B, npad); slot j holds lambda_{n0 + 1 + j}
  double* lsum;                     // adjoint: (B, npad) running sum of lambda_n
  int* fault;                       // set to 1 when a fragment stage was lost
};

__device__ __forceinline__ bool mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
  for (long long i = 0; i < WAIT_POLLS; ++i) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (ok) return true;
  }
  return false;
}

template <bool ADJ, int W>
__global__ void __launch_bounds__(32 * W, 16 / W) k_heat_roll(const RollArgs a) {
  __shared__ __align__(16) double stg[2][FRAGD];
  __shared__ uint64_t bar[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, q = lane & 3;
  const int npad = a.npad, nb = npad >> 5, nsub = 2 * nb, nfree = a.nfree;
  const long long B = a.B;
  const long long s0 = (blockIdx.x * static_cast<long long>(W) + warp) * MMA_S;
  long long sid[2];
  bool valid[2];
  double* row[2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    const long long s = s0 + 8 * mt + g;
    valid[mt] = s < B;
    sid[mt] = valid[mt] ? s : B - 1;
    row[mt] = a.X + sid[mt] * npad + 2 * q;
  }
  const double* gs[2] = {nullptr, nullptr};   // adjoint: this step's dL/du_n rows, null on steps that were not recorded
  double* urow[2];                             // forward: this step's trajectory rows
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) urow[mt] = ADJ ? nullptr : a.traj + sid[mt] * a.ld_b;
  auto set_gbar = [&](int it) {
    const int n = a.n0 + a.nt - it;
    const bool rec = ADJ && a.gbar != nullptr && n % a.gev == 0;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
      gs[mt] = rec ? a.gbar + sid[mt] * a.ldg_b + static_cast<long long>(n / a.gev - 1) * a.ldg_t : nullptr;
  };
  // forward from u0: x_0 = u0[free] into the carry, each lane the positions it reads back below (no synchronisation)
  if (!ADJ && a.u0 != nullptr) {
    for (int c0 = 2 * q; c0 < npad; c0 += 8) {
      const int n0 = c0 < nfree ? a.fnode[c0] : -1, n1 = c0 + 1 < nfree ? a.fnode[c0 + 1] : -1;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
        const double x0 = n0 >= 0 ? a.u0[sid[mt] * a.ldu0 + n0] : 0.0, x1 = n1 >= 0 ? a.u0[sid[mt] * a.ldu0 + n1] : 0.0;
        if (valid[mt]) *reinterpret_cast<double2*>(row[mt] + c0 - 2 * q) = make_double2(x0, x1);
      }
    }
  }
  // carry -> right-hand side in place: fma(m, x_n, c) (forward) / fma(m, lambda_{n+1}, gbar_n[free]) (adjoint)
  auto form_rhs = [&](int kb, Blk& R) {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int c0 = 32 * kb + 8 * nt + 2 * q;
      const double2 mm = *reinterpret_cast<const double2*>(a.mf + c0);
      if (!ADJ) {
        const double2 cc = *reinterpret_cast<const double2*>(a.cf + c0);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          R[mt][nt][0] = fma(mm.x, R[mt][nt][0], cc.x);
          R[mt][nt][1] = fma(mm.y, R[mt][nt][1], cc.y);
        }
      } else {
        const int n0 = c0 < nfree ? a.fnode[c0] : -1, n1 = c0 + 1 < nfree ? a.fnode[c0 + 1] : -1;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const double g0 = (gs[mt] && n0 >= 0) ? gs[mt][n0] : 0.0, g1 = (gs[mt] && n1 >= 0) ? gs[mt][n1] : 0.0;
          R[mt][nt][0] = fma(mm.x, R[mt][nt][0], g0);
          R[mt][nt][1] = fma(mm.y, R[mt][nt][1], g1);
        }
      }
    }
  };
  if (tid == 0) {
    mbar_init_raw(&bar[0], 1);
    mbar_init_raw(&bar[1], 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(&bar[0], FRAGD * 8u);
    bulk_g2s(stg[0], frag_src(a.Ff, a.Bf, nb, 0), FRAGD * 8u, &bar[0]);
  }
  Blk R, P = {}, acc;
  set_gbar(0);
  ld_block(row, 0, R);
  form_rhs(0, R);
  bool lost = false;
  long long G = 0;   // stage counter over the whole rollout: fragment slot G & 1, barrier parity (G >> 1) & 1
  for (int it = 0; it < a.nt; ++it) {
    for (int step = 0; step < nsub; ++step, ++G) {
      const int k = band_block(step, nb);
      __syncthreads();   // every warp has finished stage G - 1: the other slot is free (and, at G = 0, the barriers exist)
      if (tid == 0 && !(it + 1 == a.nt && step + 1 == nsub)) {   // the fragment sequence repeats every time step
        const int ns = step + 1 < nsub ? step + 1 : 0;
        mbar_arrive_expect_tx(&bar[(G + 1) & 1], FRAGD * 8u);
        bulk_g2s(stg[(G + 1) & 1], frag_src(a.Ff, a.Bf, nb, ns), FRAGD * 8u, &bar[(G + 1) & 1]);
      }
      if (!mbar_wait_bounded(&bar[G & 1], static_cast<uint32_t>((G >> 1) & 1))) lost = true;
      Blk t;
      blk_copy(t, R);
      const int knext = band_block(step + 1, nb);   // == k at the turn-around
      // the right-hand side of the next block is in flight while the two products run.  (One load per branch, and the
      // redundant step + 1 < nsub test of the turn-around below: the merged forms spill at 128 registers.)
      if (step + 1 < nsub && knext != k) {
        if (step + 1 < nb) {
          ld_block(row, knext, R);
          form_rhs(knext, R);
        } else {
          ld_block(row, knext, R);
        }
      }
      band_step(step, nb, stg[G & 1], lane, t, P, acc);
      const int jslot = a.nt - 1 - it;   // adjoint: lambda_{n0 + 1 + jslot} is this time step's result
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          P[mt][nt][0] = acc[mt][nt][0];
          P[mt][nt][1] = acc[mt][nt][1];
          if (step + 1 < nsub && knext == k) { R[mt][nt][0] = acc[mt][nt][0]; R[mt][nt][1] = acc[mt][nt][1]; }   // turn-around
          if (!valid[mt]) continue;
          const int off = 32 * k + 8 * nt;
          *reinterpret_cast<double2*>(row[mt] + off) = make_double2(acc[mt][nt][0], acc[mt][nt][1]);   // y, or the new carry
          if (step >= nb) {   // backward pass: block k of x_{n+1} / lambda_n is final
            if (!ADJ) {
              const int c0 = off + 2 * q;
              if (c0 < nfree) urow[mt][a.fnode[c0]] = acc[mt][nt][0];
              if (c0 + 1 < nfree) urow[mt][a.fnode[c0 + 1]] = acc[mt][nt][1];
            } else {
              const long long ro = sid[mt] * npad + off + 2 * q;
              *reinterpret_cast<double2*>(a.lam + static_cast<long long>(jslot) * B * npad + ro) =
                  make_double2(acc[mt][nt][0], acc[mt][nt][1]);
              double2 s = *reinterpret_cast<const double2*>(a.lsum + ro);
              s.x += acc[mt][nt][0];
              s.y += acc[mt][nt][1];
              *reinterpret_cast<double2*>(a.lsum + ro) = s;
            }
          }
        }
    }
    if (!ADJ) {   // u[d] = g on the Dirichlet nodes of this step's trajectory rows; the 4 lanes of a sample share them
      for (int d = q; d < a.n_dir; d += 4) {
        const int node = a.dir_idx[d];
        const double gv = a.dir_val[d];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          if (valid[mt]) urow[mt][node] = gv;
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) urow[mt] += a.ld_t;
    }
    if (it + 1 < a.nt) {   // block 0 of the carry is in acc: the first right-hand side block of the next step, from registers
      set_gbar(it + 1);
      blk_copy(R, acc);
      form_rhs(0, R);
    }
  }
  if (lost) atomicExch(a.fault, 1);
}

// per element: K0 (k00 k01 k02 k11 k12 k22) at kappa = 1, node ids and lambda slots (free rank, or npad: a zero)
__global__ void k_heat_tables(const MeshDev M, int npad, double* __restrict__ K0, int4* __restrict__ eidx) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= M.n_el) return;
  int n[3];
  double b[3], c[3];
  for (int i = 0; i < 3; ++i) n[i] = M.elems[3 * e + i];
  const double xi = M.nodes[2 * n[0]], yi = M.nodes[2 * n[0] + 1];
  const double xj = M.nodes[2 * n[1]], yj = M.nodes[2 * n[1] + 1];
  const double xk = M.nodes[2 * n[2]], yk = M.nodes[2 * n[2] + 1];
  const double area = 0.5 * fabs((xj - xi) * (yk - yi) - (xk - xi) * (yj - yi));
  b[0] = yj - yk; b[1] = yk - yi; b[2] = yi - yj;
  c[0] = xk - xj; c[1] = xi - xk; c[2] = xj - xi;
  const bool keep = !(area < AREA_EPS);   // degenerate elements contribute nothing to K (solver.py:120-121)
  const double den = 4.0 * area;
  const int pq[6][2] = {{0, 0}, {0, 1}, {0, 2}, {1, 1}, {1, 2}, {2, 2}};
  for (int i = 0; i < 6; ++i) {
    const int p = pq[i][0], r = pq[i][1];
    K0[6 * static_cast<size_t>(e) + i] = keep ? (b[p] * b[r] + c[p] * c[r]) / den : 0.0;
  }
  int rk[3];
  for (int i = 0; i < 3; ++i) rk[i] = M.free_rank[n[i]] >= 0 ? M.free_rank[n[i]] : npad;
  eidx[2 * e] = make_int4(n[0], n[1], n[2], 0);
  eidx[2 * e + 1] = make_int4(rk[0], rk[1], rk[2], 0);
}

__device__ __forceinline__ void cp_async8(void* s, const void* gp) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(s)), "l"(gp) : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct GradArgs {
  int n_el, nn, npad, nchunk, cs, n0;
  long long B;
  const double* u;      // state after local step j of sample b: u + b * ld_b + j * ld_t (node layout)
  long long ld_b, ld_t;
  const double* lam;    // (n_seg, B, npad)
  const double* K0;     // (n_el, 6)
  const int4* eidx;     // (n_el, 2)
  double* part;         // (n_total, nchunk, n_el)
};

// CTA (chunk c, local step j): sum over the chunk's samples of lam~^T K0_e u for every element, in sample order
__global__ void __launch_bounds__(GT) k_heat_grad(const GradArgs a) {
  extern __shared__ __align__(16) double gsm[];
  const int rowu = (a.nn + 1) & ~1, rowl = a.npad + 2, stage = rowu + rowl;
  double* acc = gsm;
  double* ring = gsm + ((a.n_el + 1) & ~1);
  const int tid = threadIdx.x, c = blockIdx.x, j = blockIdx.y;
  const long long b0 = static_cast<long long>(c) * a.cs;
  const int cnt = static_cast<int>(b0 + a.cs <= a.B ? a.cs : (a.B > b0 ? a.B - b0 : 0));
  for (int e = tid; e < a.n_el; e += GT) acc[e] = 0.0;
  if (tid < 2 * GNST) ring[(tid >> 1) * stage + rowu + a.npad + (tid & 1)] = 0.0;   // the lambda slot of Dirichlet nodes
  auto issue = [&](int i) {
    if (i < cnt) {
      double* dst = ring + (i % GNST) * stage;
      const double* su = a.u + (b0 + i) * a.ld_b + static_cast<long long>(j) * a.ld_t;
      const double* sl = a.lam + (static_cast<long long>(j) * a.B + b0 + i) * a.npad;
      for (int t = tid; t < a.nn; t += GT) cp_async8(dst + t, su + t);
      for (int t = tid; t < a.npad; t += GT) cp_async8(dst + rowu + t, sl + t);
    }
    cp_commit();   // an empty group past the end keeps the wait count uniform
  };
#pragma unroll
  for (int i = 0; i < GNST - 1; ++i) issue(i);
  for (int i = 0; i < cnt; ++i) {
    cp_wait<GNST - 2>();
    __syncthreads();   // sample i has landed for every thread, and every thread is done with the slot refilled next
    issue(i + GNST - 1);
    const double* su = ring + (i % GNST) * stage;
    const double* sl = su + rowu;
    for (int e = tid; e < a.n_el; e += GT) {
      const int4 in = a.eidx[2 * e], ir = a.eidx[2 * e + 1];
      const double2 k01 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e));
      const double2 k23 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e) + 2);
      const double2 k45 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e) + 4);
      const double u0 = su[in.x], u1 = su[in.y], u2 = su[in.z];
      const double ku0 = fma(k01.x, u0, fma(k01.y, u1, k23.x * u2));   // k00 u0 + k01 u1 + k02 u2
      const double ku1 = fma(k01.y, u0, fma(k23.y, u1, k45.x * u2));   // k01 u0 + k11 u1 + k12 u2
      const double ku2 = fma(k23.x, u0, fma(k45.x, u1, k45.y * u2));   // k02 u0 + k12 u1 + k22 u2
      acc[e] += fma(sl[ir.x], ku0, fma(sl[ir.y], ku1, sl[ir.z] * ku2));
    }
  }
  double* out = a.part + (static_cast<size_t>(a.n0 + j) * a.nchunk + c) * a.n_el;
  for (int e = tid; e < a.n_el; e += GT) out[e] = acc[e];   // each thread reads back only the sums it wrote
}

// gk[e] = -dt sum_n (sum_c part[n][c][e]): steps in ascending order, chunks in ascending order within a step
__global__ void k_heat_gsum(int n_el, int n_total, int nchunk, const double* __restrict__ part, double mdt,
                            double* __restrict__ gk) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n_el) return;
  double tot = 0.0;
  for (int n = 0; n < n_total; ++n) {
    const double* p = part + static_cast<size_t>(n) * nchunk * n_el + e;
    double r = 0.0;
    for (int c = 0; c < nchunk; ++c) r += p[static_cast<size_t>(c) * n_el];
    tot += r;
  }
  gk[e] = mdt * tot;
}

// out[0] = sum of in[0 .. n) by one CTA of 256 threads in a fixed order
__global__ void __launch_bounds__(256) k_heat_sum1(const double* __restrict__ in, int n, double* __restrict__ out) {
  __shared__ double sh[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) s += in[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if (threadIdx.x < d) sh[threadIdx.x] += sh[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sh[0];
}

inline unsigned nblk(long long n, int t) { return static_cast<unsigned>((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

size_t grad_smem(const dfe_mesh* m) {
  const size_t rowu = (static_cast<size_t>(m->dev.n_nodes) + 1) & ~static_cast<size_t>(1);
  const size_t rowl = static_cast<size_t>(dfe_band_npad(m)) + 2;
  return (((static_cast<size_t>(m->dev.n_el) + 1) & ~static_cast<size_t>(1)) + GNST * (rowu + rowl)) * sizeof(double);
}
bool heat_fits(const dfe_mesh* m) {
  return m && m->info.device >= 0 && m->dev.dim == 2 && dfe_band_supported(m) && grad_smem(m) <= GSMEM_MAX;
}
// samples per chunk of the gradient kernel: a function of B alone
int grad_cs(long long B) { return static_cast<int>(B <= 16LL * GCHUNKS ? 16 : (B + GCHUNKS - 1) / GCHUNKS); }
int grad_nchunk(long long B) { return static_cast<int>((B + grad_cs(B) - 1) / grad_cs(B)); }
// warps per CTA of the rollout kernels: the largest of 8 and 4 whose grid still covers every SM, else 2
int roll_warps(const dfe_mesh* m, long long B) {
  for (int w = 8; w > 2; w >>= 1)
    if ((B + MMA_S * w - 1) / (MMA_S * w) >= m->sm_count) return w;
  return 2;
}

int heat_enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (!heat_fits(m)) {
    dfe::set_error("%s: needs a 2-D P1 mesh with K_free of half bandwidth <= 32 and a gradient kernel within %zu bytes of "
                   "shared memory (this mesh: dim %d, band %s, %zu bytes)", who, GSMEM_MAX, m->dev.dim,
                   dfe_band_supported(m) ? "ok" : "too wide", grad_smem(m));
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}
bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <bool ADJ>
int roll_launch(const dfe_mesh* m, int warps, RollArgs a, const void* factor, cudaStream_t st, const char* who) {
  if (warps == 0) warps = roll_warps(m, a.B);
  if (warps != 2 && warps != 4 && warps != 8) {
    dfe::set_error("%s: warps must be 0 (automatic), 2, 4 or 8", who);
    return DFE_ERR_INVALID;
  }
  a.npad = dfe_band_npad(m);
  a.nfree = m->dev.n_free;
  a.n_dir = m->dev.n_dir;
  a.fnode = m->dev.free_nodes;
  a.dir_idx = m->dev.dir_idx;
  a.dir_val = m->dev.dir_val;
  dfe::band_frags(m, factor, &a.Ff, &a.Bf);
  const unsigned grid = nblk(a.B, MMA_S * warps);
  switch (warps) {
    case 8: k_heat_roll<ADJ, 8><<<grid, 256, 0, st>>>(a); break;
    case 4: k_heat_roll<ADJ, 4><<<grid, 128, 0, st>>>(a); break;
    default: k_heat_roll<ADJ, 2><<<grid, 64, 0, st>>>(a); break;
  }
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    dfe::set_error("%s: kernel launch failed: %s", who, cudaGetErrorString(e));
    return DFE_ERR_CUDA;
  }
  return DFE_OK;
}

// ---------------------------------------------------------------------------------------------- per-sample conductivity
constexpr int PSW = 4;   // warps per CTA of k_hps_roll (one warp per sample)

// vals (B, nnz_full): K_b -> A_b = fl(dt K_b), then fl(A_b + mass) on the diagonal; thread (p, b) owns row p of sample b
__global__ void k_hps_shift(const MeshDev M, long long B, double dt, const double* __restrict__ mass,
                            double* __restrict__ vals) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_nodes) return;
  for (long long b = blockIdx.y; b < B; b += gridDim.y) {
    double* vb = vals + b * M.nnz_full;
    for (int k = M.rowptr[p]; k < M.rowptr[p + 1]; ++k) {
      const double v = __dmul_rn(dt, vb[k]);   // no contraction: two roundings, as float(dt) * vals; A[diag] += mass
      vb[k] = M.col[k] == p ? __dadd_rn(v, mass[p]) : v;
    }
  }
}

// c (B, npad): c_b[r] = fl(dt F[node r]) - sum_k fl(A_b[lift_src[k]] g_k) in the mesh's dict order, zero for r >= n_free
__global__ void k_hps_cfree(const MeshDev M, long long B, int npad, double dt, const double* __restrict__ load,
                            const double* __restrict__ vals, double* __restrict__ c) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= npad) return;
  for (long long b = blockIdx.y; b < B; b += gridDim.y) {
    double v = 0.0;
    if (r < M.n_free) {
      const double* vb = vals + b * M.nnz_full;
      double lift = 0.0;
      for (int k = M.lift_ptr[r]; k < M.lift_ptr[r + 1]; ++k) lift = __dadd_rn(lift, __dmul_rn(vb[M.lift_src[k]], M.lift_g[k]));
      v = __dsub_rn(__dmul_rn(dt, load ? load[M.free_nodes[r]] : 0.0), lift);
    }
    c[b * npad + r] = v;
  }
}

struct PsRollArgs {
  int npad, nfree, n_dir, nt;       // nt: time steps of this launch
  long long B;
  const double* fac;                // (B, npad * 33) per-sample factors of k_bps_factor
  const int* fnode;
  const int* dir_idx;
  const double* dir_val;
  const double* mf;                 // (npad) lumped mass on the free rows, zero-padded
  const double* cf;                 // forward: (B, npad) c_b, zero-padded
  double* X;                        // (B, npad) carry: x_n (forward) / lambda_{n+1} (adjoint); y between the two sweeps
  const double* u0;                 // forward: (B, .) node-layout initial states, or null: X already holds x_0
  long long ldu0;
  double* traj;                     // forward: state after local step j at traj + b * ld_b + j * ld_t (node layout)
  long long ld_b, ld_t;
  const double* gbar;               // adjoint: dL/du_n at gbar + b * ldg_b + (n / gev - 1) * ldg_t when n % gev == 0
  long long ldg_b, ldg_t;
  int gev, n0;                      // adjoint: steps n0 + nt down to n0 + 1
  double* lam;                      // adjoint: (nt, B, npad); slot j holds lambda_{n0 + 1 + j}
  double* lsum;                     // adjoint: (B, npad) running sum of lambda_n
};

template <bool ADJ>
__global__ void __launch_bounds__(32 * PSW) k_hps_roll(const PsRollArgs a) {
  const int lane = threadIdx.x & 31;
  const long long b = blockIdx.x * static_cast<long long>(PSW) + (threadIdx.x >> 5);
  if (b >= a.B) return;
  const int npad = a.npad, nb = npad >> 5, n = a.nfree;
  const double* invd = a.fac + b * (static_cast<long long>(npad) * 33);
  const double* Lr = invd + npad;
  double* x = a.X + b * npad;
  if (!ADJ && a.u0 != nullptr)   // x_0 = u0[free]: each lane the rows it owns in the sweeps
    for (int i = lane; i < npad; i += 32) x[i] = i < n ? a.u0[b * a.ldu0 + a.fnode[i]] : 0.0;
  for (int it = 0; it < a.nt; ++it) {
    if (!ADJ) {
      const double* cb = a.cf + b * npad;
      double* urow = a.traj + b * a.ld_b + it * a.ld_t;
      bps_sweeps(
          invd, Lr, x, nb, lane, [&](int i) { return fma(a.mf[i], x[i], cb[i]); },
          [&](int i, double xv) {
            x[i] = xv;
            if (i < n) urow[a.fnode[i]] = xv;
          });
      for (int d = lane; d < a.n_dir; d += 32) urow[a.dir_idx[d]] = a.dir_val[d];
    } else {
      const int step = a.n0 + a.nt - it;
      const double* gs = (a.gbar != nullptr && step % a.gev == 0)
                             ? a.gbar + b * a.ldg_b + static_cast<long long>(step / a.gev - 1) * a.ldg_t
                             : nullptr;
      double* lrow = a.lam + (static_cast<long long>(a.nt - 1 - it) * a.B + b) * npad;
      double* srow = a.lsum + b * npad;
      bps_sweeps(
          invd, Lr, x, nb, lane,
          [&](int i) { return fma(a.mf[i], x[i], (gs != nullptr && i < n) ? gs[a.fnode[i]] : 0.0); },
          [&](int i, double xv) {
            x[i] = xv;
            lrow[i] = xv;
            srow[i] += xv;
          });
    }
  }
}

struct PsGradArgs {
  int n_el, npad, n_seg;
  long long B;
  const double* u;      // state after local step j of sample b: u + b * ld_b + j * ld_t (node layout)
  long long ld_b, ld_t;
  const double* lam;    // (n_seg, B, npad)
  const double* K0;     // (n_el, 6)
  const int4* eidx;     // (n_el, 2)
  double* gacc;         // (B, n_el) running sums
};

// thread (e, b): gacc[b][e] += lam~_j^T K0_e u_j for j = n_seg - 1 down to 0, one step at a time
__global__ void k_hps_grad(const PsGradArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.n_el) return;
  const int4 in = a.eidx[2 * e], ir = a.eidx[2 * e + 1];
  const double2 k01 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e));
  const double2 k23 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e) + 2);
  const double2 k45 = *reinterpret_cast<const double2*>(a.K0 + 6 * static_cast<size_t>(e) + 4);
  const int npad = a.npad;
  for (long long b = blockIdx.y; b < a.B; b += gridDim.y) {
    double acc = a.gacc[b * a.n_el + e];
    for (int j = a.n_seg - 1; j >= 0; --j) {
      const double* su = a.u + b * a.ld_b + j * a.ld_t;
      const double* sl = a.lam + (j * a.B + b) * npad;
      const double u0 = su[in.x], u1 = su[in.y], u2 = su[in.z];
      const double ku0 = fma(k01.x, u0, fma(k01.y, u1, k23.x * u2));   // k00 u0 + k01 u1 + k02 u2
      const double ku1 = fma(k01.y, u0, fma(k23.y, u1, k45.x * u2));   // k01 u0 + k11 u1 + k12 u2
      const double ku2 = fma(k23.x, u0, fma(k45.x, u1, k45.y * u2));   // k02 u0 + k12 u1 + k22 u2
      const double l0 = ir.x < npad ? sl[ir.x] : 0.0, l1 = ir.y < npad ? sl[ir.y] : 0.0, l2 = ir.z < npad ? sl[ir.z] : 0.0;
      acc += fma(l0, ku0, fma(l1, ku1, l2 * ku2));
    }
    a.gacc[b * a.n_el + e] = acc;
  }
}

// SUM = false: gk (B, n_el) = -dt gacc;  SUM = true: gk[b] = sum_e (-dt gacc[b][e]) by one CTA of 256 threads per sample in
// a fixed order (the reduction of k_heat_sum1)
template <bool SUM>
__global__ void __launch_bounds__(256) k_hps_gsum(int n_el, long long B, double mdt, const double* __restrict__ gacc,
                                                  double* __restrict__ gk) {
  if (!SUM) {
    const long long i = blockIdx.x * 256LL + threadIdx.x;
    if (i < B * n_el) gk[i] = mdt * gacc[i];
    return;
  }
  __shared__ double sh[256];
  const double* g = gacc + static_cast<long long>(blockIdx.x) * n_el;
  double s = 0.0;
  for (int i = threadIdx.x; i < n_el; i += 256) s += mdt * g[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int d = 128; d > 0; d >>= 1) {
    if (threadIdx.x < d) sh[threadIdx.x] += sh[threadIdx.x + d];
    __syncthreads();
  }
  if (threadIdx.x == 0) gk[blockIdx.x] = sh[0];
}

size_t hps_sample(const dfe_mesh* m) { return static_cast<size_t>(dfe_band_npad(m)) * 33; }   // doubles of one factor

int hps_enter(const dfe_mesh* m, const char* who, int* prev) {
  if (!m) {
    dfe::set_error("%s: mesh is null", who);
    return DFE_ERR_INVALID;
  }
  if (m->info.device < 0) {
    dfe::set_error("%s: mesh handle is host-only; no CUDA device (this library has no CPU path)", who);
    return DFE_ERR_CUDA;
  }
  if (!dfe_band_ps_supported(m)) {
    dfe::set_error("%s: needs a 2-D P1 mesh whose K_free has half bandwidth <= 32 (dfe_band_ps_supported)", who);
    return DFE_ERR_UNSUPPORTED;
  }
  DFE_CUDA_OK(cudaGetDevice(prev));
  if (*prev != m->info.device) DFE_CUDA_OK(cudaSetDevice(m->info.device));
  return DFE_OK;
}

int launch_status(const char* who) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return DFE_OK;
  dfe::set_error("%s: kernel launch failed: %s", who, cudaGetErrorString(e));
  return DFE_ERR_CUDA;
}

inline unsigned ygrid(long long B) { return static_cast<unsigned>(B < 65535 ? B : 65535); }

template <bool ADJ>
int hps_roll_launch(const dfe_mesh* m, PsRollArgs a, const void* factors, cudaStream_t st, const char* who) {
  a.npad = static_cast<int>(dfe_band_npad(m));
  a.nfree = m->dev.n_free;
  a.n_dir = m->dev.n_dir;
  a.fnode = m->dev.free_nodes;
  a.dir_idx = m->dev.dir_idx;
  a.dir_val = m->dev.dir_val;
  a.fac = static_cast<const double*>(factors) + 10 * static_cast<size_t>(m->dev.n_el);
  k_hps_roll<ADJ><<<nblk(a.B, PSW), 32 * PSW, 0, st>>>(a);
  return launch_status(who);
}

}  // namespace

extern "C" int dfe_heat_supported(const dfe_mesh* m) { return heat_fits(m) ? 1 : 0; }

extern "C" int dfe_heat_warps(const dfe_mesh* m, int64_t B) { return (heat_fits(m) && B > 0) ? roll_warps(m, B) : 0; }

extern "C" size_t dfe_heat_grad_bytes(const dfe_mesh* m, int64_t B, int64_t n_steps) {
  if (!heat_fits(m) || B < 1 || n_steps < 1) return 0;
  const size_t ne = static_cast<size_t>(m->dev.n_el);
  return (6 * ne + 4 * ne + static_cast<size_t>(n_steps) * grad_nchunk(B) * ne + ne) * sizeof(double);
}

extern "C" int dfe_heat_fwd(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0,
                            const void* factor, const double* m_free, const double* c_free, double* X, double* traj,
                            int64_t ld_b, int64_t ld_t, int warps, int32_t* fault, void* stream) {
  int prev;
  int rc = heat_enter(m, "dfe_heat_fwd", &prev);
  if (rc) return rc;
  if (!factor || !m_free || !c_free || !X || !traj || !fault || B < 1 || n_steps < 1 || n_steps > (1LL << 30) ||
      !al16(m_free) || !al16(c_free) || !al16(X)) {
    dfe::set_error("dfe_heat_fwd: null / invalid argument (m_free, c_free and X must be 16-byte aligned)");
    rc = DFE_ERR_INVALID;
  } else {
    RollArgs a{};
    a.B = B;
    a.nt = static_cast<int>(n_steps);
    a.mf = m_free;
    a.cf = c_free;
    a.X = X;
    a.u0 = u0;
    a.ldu0 = ldu0;
    a.traj = traj;
    a.ld_b = ld_b;
    a.ld_t = ld_t;
    a.fault = fault;
    rc = roll_launch<false>(m, warps, a, factor, static_cast<cudaStream_t>(stream), "dfe_heat_fwd");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_adj(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_steps, const double* gbar, int64_t ldg_b,
                            int64_t ldg_t, int64_t g_every, const void* factor, const double* m_free, double* X,
                            double* lam, double* lam_sum, int warps, int32_t* fault, void* stream) {
  int prev;
  int rc = heat_enter(m, "dfe_heat_adj", &prev);
  if (rc) return rc;
  if (!factor || !m_free || !X || !lam || !lam_sum || !fault || B < 1 || n0 < 0 || n_steps < 1 ||
      n0 + n_steps > (1LL << 30) || (gbar && g_every < 1) || !al16(m_free) || !al16(X) || !al16(lam) || !al16(lam_sum)) {
    dfe::set_error("dfe_heat_adj: null / invalid argument (m_free, X, lam and lam_sum must be 16-byte aligned)");
    rc = DFE_ERR_INVALID;
  } else {
    RollArgs a{};
    a.B = B;
    a.nt = static_cast<int>(n_steps);
    a.mf = m_free;
    a.X = X;
    a.gbar = gbar;
    a.ldg_b = ldg_b;
    a.ldg_t = ldg_t;
    a.gev = gbar ? static_cast<int>(g_every) : 1;
    a.n0 = static_cast<int>(n0);
    a.lam = lam;
    a.lsum = lam_sum;
    a.fault = fault;
    rc = roll_launch<true>(m, warps, a, factor, static_cast<cudaStream_t>(stream), "dfe_heat_adj");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_grad(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_seg, int64_t n_total, const double* u,
                             int64_t ld_b, int64_t ld_t, const double* lam, void* ws, size_t ws_bytes, void* stream) {
  int prev;
  int rc = heat_enter(m, "dfe_heat_grad", &prev);
  if (rc) return rc;
  if (!u || !lam || !ws || B < 1 || n0 < 0 || n_seg < 1 || n_seg > 65535 || n0 + n_seg > n_total) {
    dfe::set_error("dfe_heat_grad: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_heat_grad_bytes(m, B, n_total)) {
    dfe::set_error("dfe_heat_grad: workspace %zu bytes < required %zu", ws_bytes, dfe_heat_grad_bytes(m, B, n_total));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ne = m->dev.n_el;
    GradArgs a{};
    a.n_el = ne;
    a.nn = m->dev.n_nodes;
    a.npad = dfe_band_npad(m);
    a.cs = grad_cs(B);
    a.nchunk = grad_nchunk(B);
    a.n0 = static_cast<int>(n0);
    a.B = B;
    a.u = u;
    a.ld_b = ld_b;
    a.ld_t = ld_t;
    a.lam = lam;
    double* K0 = static_cast<double*>(ws);
    a.K0 = K0;
    a.eidx = reinterpret_cast<const int4*>(K0 + 6 * static_cast<size_t>(ne));
    a.part = K0 + 10 * static_cast<size_t>(ne);
    k_heat_tables<<<nblk(ne, 128), 128, 0, st>>>(m->dev, a.npad, K0, reinterpret_cast<int4*>(K0 + 6 * static_cast<size_t>(ne)));
    const size_t sm = grad_smem(m);
    cudaError_t e = cudaFuncSetAttribute(k_heat_grad, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(sm));
    if (e == cudaSuccess) {
      k_heat_grad<<<dim3(static_cast<unsigned>(a.nchunk), static_cast<unsigned>(n_seg)), GT, sm, st>>>(a);
      e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
      dfe::set_error("dfe_heat_grad: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_grad_sum(const dfe_mesh* m, int64_t B, int64_t n_total, double dt, int kappa_mode, double* gkappa,
                                 void* ws, size_t ws_bytes, void* stream) {
  int prev;
  int rc = heat_enter(m, "dfe_heat_grad_sum", &prev);
  if (rc) return rc;
  if (!gkappa || !ws || B < 1 || n_total < 1) {
    dfe::set_error("dfe_heat_grad_sum: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_SCALAR && kappa_mode != DFE_KAPPA_PER_ELEMENT) {
    dfe::set_error("dfe_heat_grad_sum: kappa_mode must be SCALAR or PER_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_heat_grad_bytes(m, B, n_total)) {
    dfe::set_error("dfe_heat_grad_sum: workspace %zu bytes < required %zu", ws_bytes, dfe_heat_grad_bytes(m, B, n_total));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ne = m->dev.n_el, nch = grad_nchunk(B);
    const double* part = static_cast<const double*>(ws) + 10 * static_cast<size_t>(ne);
    double* tmp = static_cast<double*>(ws) + (10 + static_cast<size_t>(n_total) * nch) * static_cast<size_t>(ne);
    const bool scalar = kappa_mode == DFE_KAPPA_SCALAR;
    k_heat_gsum<<<nblk(ne, 128), 128, 0, st>>>(ne, static_cast<int>(n_total), nch, part, -dt, scalar ? tmp : gkappa);
    if (scalar) k_heat_sum1<<<1, 256, 0, st>>>(tmp, ne, gkappa);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      dfe::set_error("dfe_heat_grad_sum: kernel launch failed: %s", cudaGetErrorString(e));
      rc = DFE_ERR_CUDA;
    }
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

// ---------------------------------------------------------------------------------------------- per-sample conductivity
extern "C" size_t dfe_heat_ps_factor_bytes(const dfe_mesh* m, int64_t B) {
  if (!dfe_band_ps_supported(m) || B < 1) return 0;
  return (10 * static_cast<size_t>(m->dev.n_el) + static_cast<size_t>(B) * hps_sample(m)) * sizeof(double);
}

extern "C" size_t dfe_heat_ps_workspace_bytes(const dfe_mesh* m, int64_t B) {
  if (!dfe_band_ps_supported(m) || B < 1) return 0;
  // A (B, nnz_full) doubles | bidx (npad, 33) int32
  return static_cast<size_t>(B) * m->dev.nnz_full * sizeof(double) + hps_sample(m) * sizeof(int);
}

extern "C" int dfe_heat_ps_setup(const dfe_mesh* m, int64_t B, const double* kappa, int kappa_mode, double dt,
                                 const double* mass, const double* load, void* factors, double* c_free, int32_t* status,
                                 void* ws, size_t ws_bytes, void* stream) {
  int prev;
  int rc = hps_enter(m, "dfe_heat_ps_setup", &prev);
  if (rc) return rc;
  if (!kappa || !mass || !factors || !c_free || !status || !ws || B < 1 || !al16(factors)) {
    dfe::set_error("dfe_heat_ps_setup: null / invalid argument (factors must be 16-byte aligned)");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_PER_SAMPLE && kappa_mode != DFE_KAPPA_PER_SAMPLE_ELEMENT) {
    dfe::set_error("dfe_heat_ps_setup: kappa_mode must be PER_SAMPLE or PER_SAMPLE_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else if (ws_bytes < dfe_heat_ps_workspace_bytes(m, B)) {
    dfe::set_error("dfe_heat_ps_setup: workspace %zu bytes < required %zu", ws_bytes, dfe_heat_ps_workspace_bytes(m, B));
    rc = DFE_ERR_WORKSPACE;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int np = static_cast<int>(dfe_band_npad(m)), ne = m->dev.n_el;
    double* K0 = static_cast<double*>(factors);
    double* fac = K0 + 10 * static_cast<size_t>(ne);
    double* A = static_cast<double*>(ws);
    int* bidx = reinterpret_cast<int*>(A + static_cast<size_t>(B) * m->dev.nnz_full);
    k_heat_tables<<<nblk(ne, 128), 128, 0, st>>>(m->dev, np, K0, reinterpret_cast<int4*>(K0 + 6 * static_cast<size_t>(ne)));
    dfe::band_ps_assemble(m, B, kappa, kappa_mode == DFE_KAPPA_PER_SAMPLE_ELEMENT, A, st);
    k_hps_shift<<<dim3(nblk(m->dev.n_nodes, 128), ygrid(B)), 128, 0, st>>>(m->dev, B, dt, mass, A);
    k_hps_cfree<<<dim3(nblk(np, 128), ygrid(B)), 128, 0, st>>>(m->dev, B, np, dt, load, A, c_free);
    dfe::band_ps_factor(m, B, A, m->dev.nnz_full, bidx, fac, status, st);
    rc = launch_status("dfe_heat_ps_setup");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_ps_fwd(const dfe_mesh* m, int64_t B, int64_t n_steps, const double* u0, int64_t ldu0,
                               const void* factors, const double* m_free, const double* c_free, double* X, double* traj,
                               int64_t ld_b, int64_t ld_t, void* stream) {
  int prev;
  int rc = hps_enter(m, "dfe_heat_ps_fwd", &prev);
  if (rc) return rc;
  if (!factors || !m_free || !c_free || !X || !traj || B < 1 || n_steps < 1 || n_steps > (1LL << 30)) {
    dfe::set_error("dfe_heat_ps_fwd: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else {
    PsRollArgs a{};
    a.B = B;
    a.nt = static_cast<int>(n_steps);
    a.mf = m_free;
    a.cf = c_free;
    a.X = X;
    a.u0 = u0;
    a.ldu0 = ldu0;
    a.traj = traj;
    a.ld_b = ld_b;
    a.ld_t = ld_t;
    rc = hps_roll_launch<false>(m, a, factors, static_cast<cudaStream_t>(stream), "dfe_heat_ps_fwd");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_ps_adj(const dfe_mesh* m, int64_t B, int64_t n0, int64_t n_steps, const double* gbar,
                               int64_t ldg_b, int64_t ldg_t, int64_t g_every, const void* factors, const double* m_free,
                               double* X, double* lam, double* lam_sum, void* stream) {
  int prev;
  int rc = hps_enter(m, "dfe_heat_ps_adj", &prev);
  if (rc) return rc;
  if (!factors || !m_free || !X || !lam || !lam_sum || B < 1 || n0 < 0 || n_steps < 1 || n0 + n_steps > (1LL << 30) ||
      (gbar && g_every < 1)) {
    dfe::set_error("dfe_heat_ps_adj: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else {
    PsRollArgs a{};
    a.B = B;
    a.nt = static_cast<int>(n_steps);
    a.mf = m_free;
    a.X = X;
    a.gbar = gbar;
    a.ldg_b = ldg_b;
    a.ldg_t = ldg_t;
    a.gev = gbar ? static_cast<int>(g_every) : 1;
    a.n0 = static_cast<int>(n0);
    a.lam = lam;
    a.lsum = lam_sum;
    rc = hps_roll_launch<true>(m, a, factors, static_cast<cudaStream_t>(stream), "dfe_heat_ps_adj");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_ps_grad(const dfe_mesh* m, int64_t B, int64_t n_seg, const void* factors, const double* u,
                                int64_t ld_b, int64_t ld_t, const double* lam, double* gacc, void* stream) {
  int prev;
  int rc = hps_enter(m, "dfe_heat_ps_grad", &prev);
  if (rc) return rc;
  if (!factors || !u || !lam || !gacc || B < 1 || n_seg < 1 || n_seg > (1LL << 30)) {
    dfe::set_error("dfe_heat_ps_grad: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else {
    const int ne = m->dev.n_el;
    PsGradArgs a{};
    a.n_el = ne;
    a.npad = static_cast<int>(dfe_band_npad(m));
    a.n_seg = static_cast<int>(n_seg);
    a.B = B;
    a.u = u;
    a.ld_b = ld_b;
    a.ld_t = ld_t;
    a.lam = lam;
    a.K0 = static_cast<const double*>(factors);
    a.eidx = reinterpret_cast<const int4*>(a.K0 + 6 * static_cast<size_t>(ne));
    a.gacc = gacc;
    k_hps_grad<<<dim3(nblk(ne, 128), ygrid(B)), 128, 0, static_cast<cudaStream_t>(stream)>>>(a);
    rc = launch_status("dfe_heat_ps_grad");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}

extern "C" int dfe_heat_ps_grad_sum(const dfe_mesh* m, int64_t B, double dt, int kappa_mode, const double* gacc,
                                    double* gkappa, void* stream) {
  int prev;
  int rc = hps_enter(m, "dfe_heat_ps_grad_sum", &prev);
  if (rc) return rc;
  if (!gacc || !gkappa || B < 1 || B > 0x7fffffffLL) {
    dfe::set_error("dfe_heat_ps_grad_sum: null / invalid argument");
    rc = DFE_ERR_INVALID;
  } else if (kappa_mode != DFE_KAPPA_PER_SAMPLE && kappa_mode != DFE_KAPPA_PER_SAMPLE_ELEMENT) {
    dfe::set_error("dfe_heat_ps_grad_sum: kappa_mode must be PER_SAMPLE or PER_SAMPLE_ELEMENT");
    rc = DFE_ERR_INVALID;
  } else {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int ne = m->dev.n_el;
    if (kappa_mode == DFE_KAPPA_PER_SAMPLE) k_hps_gsum<true><<<static_cast<unsigned>(B), 256, 0, st>>>(ne, B, -dt, gacc, gkappa);
    else k_hps_gsum<false><<<nblk(B * ne, 256), 256, 0, st>>>(ne, B, -dt, gacc, gkappa);
    rc = launch_status("dfe_heat_ps_grad_sum");
  }
  if (prev != m->info.device) cudaSetDevice(prev);
  return rc;
}
