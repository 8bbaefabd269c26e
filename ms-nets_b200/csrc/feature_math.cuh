// feature_math.cuh -- channel normalisation and AML arithmetic shared by every
// kernel that emits feature planes (features.cu, ms_fused.cu, fte.cu).
#pragma once
#include "common.cuh"

namespace msn {

// ch0 clip(census,0,120)/120 ; ch1 (1+clip(ncc,-1,1))/2 ; ch2/ch3 clip(.,0,8192)/8192
// in IEEE fp32 exactly as NumPy evaluates them (cbmv_generator.py:283-287).
// The division by 120 is a true division (not a reciprocal multiply) so channel 0
// is bit-exact; /2 and /8192 are exact power-of-two scalings.  fill -> 1.0.
__device__ __forceinline__ float normalise_cost(float v, int matcher) {
  if (matcher == 0) return __fdiv_rn(fminf(fmaxf(v, 0.f), 120.f), 120.f);
  // One instruction each (FFMA.SAT / FMUL.SAT), bit-identical to the clip-then-scale forms:
  //  (1 + clip(v,-1,1)) * 0.5: for |v| <= 1 the sum 1 + v is rounded once and the halving is exact, so it
  //  equals round(0.5 v + 0.5) = fma(v, 0.5, 0.5); outside [-1,1] both forms give exactly 0 or 1.
  //  clip(v,0,8192) / 8192: the scaling by 2^-13 is exact, so clipping before or after it is the same.
  if (matcher == 1) return __saturatef(__fmaf_rn(v, 0.5f, 0.5f));
  return __saturatef(__fmul_rn(v, 1.0f / 8192.f));
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// AML term expf(-(c-m)^2 / sigma) = 2^(-(c-m)^2 * log2(e)/sigma)   (featextract.cpp:444-452).
// FAST mode (default): the SFU ex2 (rel. error ~2^-22) and a reciprocal multiply; the sum is replayed in the
// reference's order.  Stated bound, checked in tests/: |AML - reference| <= 2e-6 on outputs in [0,1] (1.2e-5
// on rare degenerate rows, tests/_synth.py).
// EXACT mode (msn_set_aml_exact(1)): the reference's own fp32 operations -- (c-m), its square, the IEEE division
// by sigma, glibc's expf replayed bit for bit (expf_glibc below), the sequential sum, the IEEE division by the
// denominator -- so AML is BIT-EXACT.  The mode travels in the sign of the scale: k > 0 is log2(e)/sigma,
// k < 0 is -sigma.
extern int g_aml_exact;   // capi.cu
inline float aml_scale(float sigma) { return g_aml_exact ? -sigma : 1.4426950408889634f / sigma; }

// glibc 2.27+ expf (sysdeps/ieee754/flt-32/e_expf.c, the Arm optimized-routines algorithm): exp(x) = 2^(k/32) *
// 2^(r/32), k = round(x * 32/ln2), the fraction by a cubic in fp64, the power of two from a 32-entry table whose
// exponent field is patched.  x86-64 glibc dispatches to its FMA build (e_expf-fma), in which the compiler has
// contracted every multiply-add of the source -- the rounding shift and the remainder r included; that exact
// sequence is replayed here with fp64 FMAs.  Checked against the libm of this image for EVERY negative float
// down to -104 (1 120 927 745 inputs, oracle/check_expf.c): 0 mismatches; without the contractions 1.
static __device__ const unsigned long long kExp2fTab[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull};
static __device__ __noinline__ float expf_glibc(float x) {   // x <= 0 (the AML argument); -inf and large negatives -> 0
  if (!(x >= -0x1.9fe368p6f)) return 0.0f;
  constexpr double N = 32.0;
  constexpr double InvLn2N = 0x1.71547652b82fep+0 * N, SHIFT = 0x1.8p+52;
  constexpr double C0 = 0x1.c6af84b912394p-5 / N / N / N, C1 = 0x1.ebfce50fac4f3p-3 / N / N, C2 = 0x1.62e42ff0c52d6p-1 / N;
  const double xd = (double)x;
  double kd = __fma_rn(InvLn2N, xd, SHIFT);
  const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, SHIFT);
  const double r = __fma_rn(InvLn2N, xd, -kd);
  const unsigned long long t = kExp2fTab[ki & 31ull] + (ki << 47);
  const double s = __longlong_as_double((long long)t);
  const double z = __fma_rn(C0, r, C1);
  const double r2 = __dmul_rn(r, r);
  double y = __fma_rn(C2, r, 1.0);
  y = __fma_rn(z, r2, y);
  y = __dmul_rn(y, s);
  return __double2float_rn(y);
}

__device__ __forceinline__ float aml_e_fast(float c, float m, float k) {
  const float t = c - m;
  return ex2_approx(-(t * t) * k);
}
__device__ __forceinline__ float aml_e_exact(float c, float m, float sigma) {
  const float t = __fsub_rn(c, m);
  return expf_glibc(__fdiv_rn(-__fmul_rn(t, t), sigma));
}
__device__ __forceinline__ float aml_e(float c, float m, float k) {
  return (k < 0.f) ? aml_e_exact(c, m, -k) : aml_e_fast(c, m, k);
}
// what multiplies (fast) / divides (exact) the exponentials of a row with denominator `den`
__device__ __forceinline__ float aml_row_scale(float den, bool has_cost, float k) {
  if (k < 0.f) return has_cost ? den : INFINITY;          // e / inf = 0: (min == fill) ? 0 : ..., featextract.cpp:451
  return has_cost ? 1.0f / den : 0.f;
}
__device__ __forceinline__ float aml_apply(float e, float row_scale, float k) {
  return (k < 0.f) ? __fdiv_rn(e, row_scale) : e * row_scale;
}

}  // namespace msn
