// Correctly rounded divisions without the division instruction (included inside an anonymous namespace).
//
// Correctly rounded a / b from y = RN(1 / b) with two Markstein corrections (fma residuals are exact): the first makes
// the quotient faithful (error 2^-106 before its rounding), the second then rounds it correctly (Markstein 1990; round
// to nearest, no under/overflow — the callers guard the range and fall back to the division instruction outside it).
// A double-precision division costs ~25 FP64 issue slots on sm_100; sharing one reciprocal between the entries of an
// element matrix (or using a constant one) takes the assembly kernels from FP64-bound to memory-bound.  Same bits as
// __ddiv_rn — the kernels that use these must reproduce the reference's dense K and F bit for bit.
#pragma once

__device__ __forceinline__ double div_markstein(double a, double b, double y) {
  const double q0 = __dmul_rn(a, y);
  if (a == 0.0) return q0;                       // keeps the sign of a zero numerator
  const double q1 = fma(fma(-b, q0, a), y, q0);
  return fma(fma(-b, q1, a), y, q1);
}
__device__ __forceinline__ bool mid_range(double v) { return fabs(v) > 1e-140 && fabs(v) < 1e140; }
__device__ __forceinline__ double div3(double a) {   // a / 3.0, correctly rounded
  constexpr double third = 0.333333333333333314829616256247;   // RN(1/3)
  return (a == 0.0 || mid_range(a)) ? div_markstein(a, 3.0, third) : __ddiv_rn(a, 3.0);
}

// The load term of one P1 triangle at node p (solver.py:143-145): fl(fl(area / 3) * fl(((f_i + f_j) + f_k) / 3)), with
// area3 = fl(area / 3).  assemble_row, k_band_rhs_fwd and the heat-source kernels (dfe_heat.cu) all form F with this one
// function; FAST takes the division by 3 through div3 (same bits, no division instruction).
template <bool FAST = false>
__device__ __forceinline__ double p1_load_term(double area3, double fi, double fj, double fk) {
  const double s = __dadd_rn(__dadd_rn(fi, fj), fk);
  return __dmul_rn(area3, FAST ? div3(s) : __ddiv_rn(s, 3.0));
}
