// Grid-wide fixed-order reduction (a sum, or a max) of two doubles for a cooperative (co-resident) launch, fused with the
// grid barrier the phases of a persistent solver need anyway.  Included inside an anonymous namespace by dfe_pcg.cu and
// dfe_mg.cu.
//
// *Data-as-flag*: every CTA release-stores its two partial results into its slot of the epoch's buffer (pre-set to an
// all-ones sentinel), warp 0 of every CTA polls all G slots with relaxed loads and adds them in a fixed order
// (lane-strided, then a butterfly), one acquire fence, one CTA barrier.  No atomic, no separate counter, no second
// read of a partials array: one L2 round trip after the last CTA arrives.  Three buffers rotate; a CTA resets its own
// slot of epoch E-2 just before it publishes epoch E (everybody finished reading E-2 before publishing E-1, which this
// CTA has seen complete), and the release orders the reset before the publication.
//
// Every poll is bounded (~2 s): a CTA that waits longer raises the global abort word, every poller that sees the word
// leaves, and the callers end their loops with status 7 instead of hanging the GPU.
#pragma once

constexpr unsigned long long SENTQ = 0xFFFFFFFFFFFFFFFFull;
__device__ __forceinline__ unsigned long long as_bits(double v) {
  const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(v));
  return u == SENTQ ? 0x7FF8000000000000ull : u;   // a NaN that happens to carry the sentinel payload
}

struct GridSync {
  double* slots;        // [3 epochs][gridDim.x][2], pre-set to the sentinel (0xFF bytes)
  int* abort_flag;      // global, zeroed before the launch
  int backoff;          // cycles an early arriver waits between two polls of a slot
};

__device__ __forceinline__ bool grid_aborted(const GridSync& gs) {
  return *reinterpret_cast<volatile int*>(gs.abort_flag) != 0;
}

// The combine steps: a + b (fixed order, so bit-reproducible) and fmax (exact in any order; drops a NaN).
struct SumOp {
  __device__ __forceinline__ static double f(double a, double b) { return a + b; }
};
struct MaxOp {   // for non-negative values: 0 is the identity
  __device__ __forceinline__ static double f(double a, double b) { return fmax(a, b); }
};

// Op::f-reductions of `v0` and `v1` over the whole grid; every thread of every CTA returns the same bits.  Doubles as the
// grid barrier between phases (all global writes of every CTA before the call are visible after it).  `sh`: 2 * NW + 2
// doubles.
template <int NW, class Op>
__device__ __forceinline__ void grid_reduce2(const GridSync& gs, unsigned int& epoch, double& v0, double& v1, double* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int G = gridDim.x;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    v0 = Op::f(v0, __shfl_xor_sync(0xffffffffu, v0, d));
    v1 = Op::f(v1, __shfl_xor_sync(0xffffffffu, v1, d));
  }
  if (lane == 0) { sh[2 * warp] = v0; sh[2 * warp + 1] = v1; }
  __syncthreads();
  ++epoch;
  if (warp == 0) {
    double a = 0.0, b = 0.0;
    for (int w = lane; w < NW; w += 32) { a = Op::f(a, sh[2 * w]); b = Op::f(b, sh[2 * w + 1]); }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      a = Op::f(a, __shfl_xor_sync(0xffffffffu, a, d));
      b = Op::f(b, __shfl_xor_sync(0xffffffffu, b, d));
    }
    double* cur = gs.slots + static_cast<size_t>(epoch % 3) * 2 * G;
    if (lane == 0) {
      unsigned long long* old = reinterpret_cast<unsigned long long*>(gs.slots + static_cast<size_t>((epoch + 1) % 3) * 2 * G) + 2 * blockIdx.x;
      asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(old), "l"(SENTQ), "l"(SENTQ) : "memory");
      asm volatile("st.release.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(cur + 2 * blockIdx.x), "l"(as_bits(a)), "l"(as_bits(b)) : "memory");
    }
    // poll: a lane owns slots lane, lane + 32, ... (up to NSL of them per trip).  All loads of a trip are issued before
    // the first one is examined, so a trip costs ONE L2 round trip whatever the grid size — polling the slots one after
    // the other made the barrier cost (G / 32) round trips, 3.5 us at 148 CTAs.
    constexpr int NSL = 5;
    double sa = 0.0, sb = 0.0;
    const long long t_start = clock64();
    int spins = 0;
    for (int i0 = lane; i0 < G; i0 += 32 * NSL) {
      unsigned long long ua[NSL], ub[NSL];
      unsigned pending = 0;
#pragma unroll
      for (int k = 0; k < NSL; ++k)
        if (i0 + 32 * k < G) pending |= 1u << k;
      while (pending) {
#pragma unroll
        for (int k = 0; k < NSL; ++k)
          if (pending & (1u << k))
            asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(ua[k]), "=l"(ub[k]) : "l"(cur + 2 * (i0 + 32 * k)) : "memory");
#pragma unroll
        for (int k = 0; k < NSL; ++k)
          if ((pending & (1u << k)) && ua[k] != SENTQ && ub[k] != SENTQ) pending &= ~(1u << k);
        if (pending) {
          // early arrivers back off for ~250 cycles (a busy wait on the clock, not __nanosleep, which oversleeps by
          // microseconds on B200): hundreds of spinning lanes on a handful of L2 lines delay the stores they wait for
          const long long t0 = clock64();
          while (clock64() - t0 < gs.backoff) {}
          // ~2 s: a lost CTA / protocol bug must not hang the GPU (the abort word is looked at every 256 trips only:
          // it is one more L2 round trip)
          if (((++spins & 255) == 0) && (t0 - t_start > 4000000000ll || grid_aborted(gs))) {
            *reinterpret_cast<volatile int*>(gs.abort_flag) = 1;
#pragma unroll
            for (int k = 0; k < NSL; ++k)
              if (pending & (1u << k)) ua[k] = ub[k] = 0ull;
            pending = 0;
          }
        }
      }
#pragma unroll
      for (int k = 0; k < NSL; ++k)   // fixed order: slot index ascending within the lane
        if (i0 + 32 * k < G) {
          sa = Op::f(sa, __longlong_as_double(static_cast<long long>(ua[k])));
          sb = Op::f(sb, __longlong_as_double(static_cast<long long>(ub[k])));
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      sa = Op::f(sa, __shfl_xor_sync(0xffffffffu, sa, d));
      sb = Op::f(sb, __shfl_xor_sync(0xffffffffu, sb, d));
    }
    // (the butterfly above made every lane's polls complete; one fence, then the CTA barrier, as a grid barrier does)
    __syncwarp();
    if (lane == 0) {
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
      sh[2 * NW] = sa;
      sh[2 * NW + 1] = sb;
    }
  }
  __syncthreads();
  v0 = sh[2 * NW];
  v1 = sh[2 * NW + 1];
}

// Sums of `v0` and `v1` over the whole grid (the reduction every solver phase ends with).
template <int NW>
__device__ __forceinline__ void grid_sum2(const GridSync& gs, unsigned int& epoch, double& v0, double& v1, double* sh) {
  grid_reduce2<NW, SumOp>(gs, epoch, v0, v1, sh);
}

// Largest of the non-negative `v` over the whole grid; every thread of every CTA returns the same value.
template <int NW>
__device__ __forceinline__ double grid_max(const GridSync& gs, unsigned int& epoch, double v, double* sh) {
  double unused = 0.0;
  grid_reduce2<NW, MaxOp>(gs, epoch, v, unused, sh);
  return v;
}

template <int NW>
__device__ __forceinline__ void grid_barrier(const GridSync& gs, unsigned int& epoch, double* sh) {
  double a = 0.0, b = 0.0;
  grid_sum2<NW>(gs, epoch, a, b, sh);
}
