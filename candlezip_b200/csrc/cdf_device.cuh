// Device-side CDF arithmetic shared by cdf_kernels.cu and exec.cu (see cdf_kernels.cu for the design notes).
#pragma once
#include "cz_common.cuh"

namespace czk {

__constant__ uint64_t c_exp2f_tab[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull,
};

// The 32-entry table is replicated per lane in shared memory as 64-bit words ([entry][lane], exp_tab64_init in cdf_fast.cuh) so a
// warp's 32 data-dependent lookups never bank-conflict.
struct ExpTab64 {
  const uint64_t *t;  // base + lane
  __device__ __forceinline__ uint64_t load(uint32_t entry) const { return t[entry << 5]; }
};

// Branch-free: every lane always evaluates the polynomial and the underflow case is a select at the end (a divergent
// early-out costs a BSSY/BSYNC pair per element in the unrolled column walk, profiles/ncu_summary_r01.md).
// DOMAIN: x <= 0 or NaN.  Every caller passes logit - max(logits) (src/main.rs:786-789), so glibc's overflow branch
// (x > 88.72 -> +inf) can never be taken and is not evaluated; +inf - +inf = NaN propagates through the polynomial.
template <class Tab>
__device__ __forceinline__ float cz_expf(float x, const Tab &tab) {
  const double inv_ln2_n = 0x1.71547652b82fep+0 * 32;
  const double shift = 0x1.8p+52;
  const double c0 = 0x1.c6af84b912394p-5 / 32 / 32 / 32;
  const double c1 = 0x1.ebfce50fac4f3p-3 / 32 / 32;
  const double c2 = 0x1.62e42ff0c52d6p-1 / 32;
  double xd = (double)x;
  double z = __dmul_rn(inv_ln2_n, xd);
  double kd = __dadd_rn(z, shift);
  uint64_t ki = (uint64_t)__double_as_longlong(kd);
  kd = __dsub_rn(kd, shift);
  double r = __fma_rn(inv_ln2_n, xd, -kd);
  uint64_t t = tab.load((uint32_t)(ki & 31));
  t += ki << 47;
  double s = __longlong_as_double((long long)t);
  double p = __fma_rn(c0, r, c1);
  double r2 = __dmul_rn(r, r);
  double y = __fma_rn(c2, r, 1.0);
  y = __fma_rn(p, r2, y);
  y = __dmul_rn(y, s);
  float out = __double2float_rn(y);
  out = (x < -0x1.9fe368p6f) ? 0.0f : out;  // underflow to zero
  return out;
}

// floor(acc * 2^30) clamped to [0, 2^30]  (src/main.rs:813-815; NaN -> 0 like Rust's `as i64`)
__device__ __forceinline__ uint32_t quant(double acc) {
  double f = __dmul_rn(acc, 1073741824.0);
  if (!(f == f)) return 0u;
  if (f >= 1073741824.0) return CZ_AC_CDF_TOTAL;
  if (f <= 0.0) return 0u;
  return (uint32_t)__double2ll_rd(f);
}

// a / b correctly rounded, given y = __drcp_rn(b); a >= 0, b > 0, all quantities (and the residuals) in the normal range.
__device__ __forceinline__ double cz_div_rcp(double a, double b, double y) {
  const double q0 = __dmul_rn(a, y);
  const double r0 = __fma_rn(-b, q0, a);
  const double q1 = __fma_rn(r0, y, q0);
  const double r1 = __fma_rn(-b, q1, a);
  return __fma_rn(r1, y, q1);
}
// divisors for which cz_div_rcp is used: finite, and far from the ends of the exponent range (S in [1, V], norm and sum2 near 1)
__device__ __forceinline__ bool cz_div_rcp_ok(double b) { return b >= 0x1p-64 && b <= 0x1p64; }

enum { OP_BOUNDS = 0, OP_SEARCH = 1, OP_XE = 2 };

#define CZ_P_FLOOR 0x1p-29 /* ac_p_min(): src/main.rs:235-238 */

// status bits written to *err (OR-ed)
#define CZ_DEVERR_NAN 1
#define CZ_DEVERR_SYM 2

// order-preserving int <-> float mapping used for the column max produced by the LM-head GEMM epilogue
__device__ __forceinline__ float colmax_decode(int v) {
  v ^= (v >> 31) & 0x7fffffff;
  return __int_as_float(v);
}

}  // namespace czk
