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

// The 32-entry table is replicated per lane in shared memory ([entry][lane], lo and hi words separately) so a
// warp's 32 data-dependent lookups never bank-conflict.
struct ExpTab {
  const uint32_t *lo;
  const uint32_t *hi;
  int lane;
  __device__ __forceinline__ uint64_t load(uint32_t entry) const {
    const int idx = ((int)entry << 5) + lane;
    return ((uint64_t)hi[idx] << 32) | (uint64_t)lo[idx];
  }
};
// the same table as 64-bit words [entry][lane] (cdf_fast.cuh)
struct ExpTab64 {
  const uint64_t *t;  // base + lane
  __device__ __forceinline__ uint64_t load(uint32_t entry) const { return t[entry << 5]; }
};

__device__ __forceinline__ void exp_tab_init(uint32_t *s_lo, uint32_t *s_hi) {
  for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) {
    uint64_t t = c_exp2f_tab[i >> 5];
    s_lo[i] = (uint32_t)t;
    s_hi[i] = (uint32_t)(t >> 32);
  }
  __syncthreads();
}

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

// Column walker shared by the stand-alone CDF kernels (cdf_kernels.cu) and the fused decode step (exec.cu).
// MUST be called by all 32 lanes of a warp (inactive lanes pass a clamped, valid column and active=false).
// p points at logits[0][col]; element v of the column is p[v * ld].
// order-preserving int <-> float mapping used for the column max produced by the LM-head GEMM epilogue
__device__ __forceinline__ float colmax_decode(int v) {
  v ^= (v >> 31) & 0x7fffffff;
  return __int_as_float(v);
}

// Ascending walk over elements [0, n) of one column with the loads software-pipelined: the next group of CDF_GRP
// values is already in flight (registers) while the current group is consumed, and an L2 prefetch runs CDF_PF rows
// ahead.  Consecutive rows of a column are ld*4 bytes apart (a new DRAM page every row), so without this the kernel is
// bound by memory latency x the few loads a warp has in flight, not by bandwidth.  f(v, x) returns false to stop the
// lane; the walk ends when every lane of the warp has stopped (keeps the warp converged for the callers' shuffles).
constexpr int CDF_GRP = 8;
constexpr int CDF_PF = 48;
// NC: loads go through the read-only path (__ldg).  NC = false is for a column that this thread rewrites in place between passes
// (RWKV literals mode caches exp(l - max) in the logit's slot): ordinary loads, which see the thread's own earlier stores.
template <bool NC = true, class F>
__device__ __forceinline__ void cdf_walk(const float *p, size_t ld, int n, F f) {
  auto ldv = [&](size_t off) -> float { return NC ? __ldg(p + off) : p[off]; };
  float cur[CDF_GRP], nxt[CDF_GRP];
#pragma unroll
  for (int k = 0; k < CDF_GRP; k++) cur[k] = k < n ? ldv((size_t)k * ld) : 0.f;
  bool go = true;
  int v0 = 0;
  // main loop, part 1: the current and the next group AND the prefetched rows are in range -> no bounds checks at all
  for (; v0 + CDF_PF + CDF_GRP <= n; v0 += CDF_GRP) {
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      nxt[k] = ldv((size_t)(v0 + CDF_GRP + k) * ld);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p + (size_t)(v0 + CDF_PF + k) * ld));
    }
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      if (go) go = f(v0 + k, cur[k]);
      cur[k] = nxt[k];
    }
    if (!__any_sync(0xffffffffu, go)) return;
  }
  // part 2 (the last CDF_PF rows): everything to come is already in L2 or on its way
  for (; v0 + 2 * CDF_GRP <= n; v0 += CDF_GRP) {
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) nxt[k] = ldv((size_t)(v0 + CDF_GRP + k) * ld);
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      if (go) go = f(v0 + k, cur[k]);
      cur[k] = nxt[k];
    }
    if (!__any_sync(0xffffffffu, go)) return;
  }
  // tail: at most two groups, checked
  for (; v0 < n; v0 += CDF_GRP) {
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      const int v = v0 + CDF_GRP + k;
      nxt[k] = v < n ? ldv((size_t)v * ld) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      if (go && v0 + k < n) go = f(v0 + k, cur[k]);
      cur[k] = nxt[k];
    }
    if (!__any_sync(0xffffffffu, go)) break;
  }
}

// have_max: the column max was already computed (exactly) by the producer; otherwise pass A below finds it.
// MUST be called by all 32 lanes of a warp (inactive lanes pass a clamped, valid column and active=false).
// p points at logits[0][col]; element v of the column is p[v * ld].
template <int MODE, int OP>
__device__ __forceinline__ void cdf_col(const float *__restrict__ p_in, size_t ld, int V, uint32_t arg, bool active,
                                        const ExpTab &tab, uint32_t &sym_out, uint32_t &lo_out, uint32_t &hi_out,
                                        double &xe_out, int &errbits, bool have_max = false, float known_max = 0.f) {
  // RWKV literals mode walks the column five times (S, norm, sum2, prefix; src/main.rs:758-782): the first pass leaves
  // e_v = expf(l_v - max) in the logit's slot (the logits are scratch, and each column belongs to one thread), so the later passes
  // read e_v instead of re-evaluating the 24-instruction expf.  Same values, same order: bit-identical results.
  // NOT for OP_SEARCH: the stepwise RWKV decoder keeps a stream's logits column across steps while it decodes literal bytes.
  constexpr bool kCache = MODE == CZ_CDF_RWKV_LITERALS && OP != OP_SEARCH;
  float *pw = const_cast<float *>(p_in);
  const float *p = kCache ? pw : p_in;  // (cached mode: no load may go through the read-only path)
  const int n_sym = MODE == CZ_CDF_RWKV_LITERALS ? V + 256 : V;
  sym_out = 0;
  lo_out = 0;
  hi_out = 0;
  xe_out = 0.0;
  // pass A: max (f32, NaN-ignoring exactly like `if v > max`)
  float mx = __int_as_float(0xff800000);
  if (have_max) {
    mx = known_max;
  } else {
    cdf_walk<!kCache>(p, ld, V, [&](int, float x) {
      if (x > mx) mx = x;
      return true;
    });
  }
  // pass B: S = sum_i (f64)expf(l_i - max), sequential
  double S = 0.0;
  cdf_walk<!kCache>(p, ld, V, [&](int v, float x) {
    const float e = cz_expf(__fsub_rn(x, mx), tab);
    if (kCache && active) pw[(size_t)v * ld] = e;  // (inactive lanes shadow a valid column: they must not write)
    S = __dadd_rn(S, (double)e);
    return true;
  });
  if (!(S == S) && active) errbits |= CZ_DEVERR_NAN;
  // e_v from a value read after pass B
  auto ex = [&](float x) -> float { return kCache ? x : cz_expf(__fsub_rn(x, mx), tab); };

  double norm = 1.0, sum2 = 1.0;
  const double scale = 1.0 - 256.0 * CZ_P_FLOOR;
  const bool uniform = (MODE == CZ_CDF_SMOLLM && OP != OP_XE) && (S <= 0.0);  // src/main.rs:794-798
  const double uni = 1.0 / (double)V;

  // the floored SmolLM pdf: what OP_XE evaluates for every SmolLM mode, and what CZ_CDF_SMOLLM_FLOOR codes with
  constexpr bool kFloorPdf = OP == OP_XE || MODE == CZ_CDF_SMOLLM_FLOOR;
  if (MODE == CZ_CDF_RWKV_LITERALS || kFloorPdf) {
    // softmax_pdf_floor: norm = sum_i max(e_i / S, floor)   (src/main.rs:763-764)
    double acc = 0.0;
    cdf_walk<!kCache>(p, ld, V, [&](int, float x) {
      const double q = __ddiv_rn((double)ex(x), S);
      acc = __dadd_rn(acc, fmax(q, CZ_P_FLOOR));
      return true;
    });
    norm = acc;
  }
  if (MODE == CZ_CDF_RWKV_LITERALS) {
    // combined_pdf_with_literals: sum2 over V scaled entries + 256 literal entries (src/main.rs:773-779)
    double acc = 0.0;
    cdf_walk<!kCache>(p, ld, V, [&](int, float x) {
      double q = __ddiv_rn((double)ex(x), S);
      q = __ddiv_rn(fmax(q, CZ_P_FLOOR), norm);
      acc = __dadd_rn(acc, __dmul_rn(q, scale));
      return true;
    });
    for (int j = 0; j < 256; j++) acc = __dadd_rn(acc, CZ_P_FLOOR);
    sum2 = acc;
  }

  // final pdf entry for vocab element v (< V) with logit x (cached mode: x is already e_v)
  auto pdf_vocab = [&](float x) -> double {
    if (MODE == CZ_CDF_RWKV_LITERALS) {
      double q = __ddiv_rn((double)ex(x), S);
      q = __dmul_rn(__ddiv_rn(fmax(q, CZ_P_FLOOR), norm), scale);
      return sum2 > 0.0 ? __ddiv_rn(q, sum2) : q;
    } else if (kFloorPdf) {
      const double q = __ddiv_rn((double)ex(x), S);
      return __ddiv_rn(fmax(q, CZ_P_FLOOR), norm);
    } else {
      if (uniform) return uni;
      return __ddiv_rn((double)ex(x), S);
    }
  };
  const double pdf_literal = sum2 > 0.0 ? __ddiv_rn(CZ_P_FLOOR, sum2) : CZ_P_FLOOR;  // RWKV literal symbols v >= V

  if (OP == OP_XE) {
    double pr = CZ_P_FLOOR;  // pdf.get(sym).unwrap_or(ac_p_min())
    if ((int)arg < V) pr = pdf_vocab(kCache ? p[(size_t)arg * ld] : __ldg(p + (size_t)arg * ld));
    else if ((int)arg < n_sym) pr = pdf_literal;
    pr = fmax(pr, 1e-300);
    xe_out = -log2(pr);
    return;
  }

  if (OP == OP_BOUNDS) {
    uint32_t sym = arg;
    bool sym_bad = false;
    if ((int)sym >= n_sym) {
      if (active) errbits |= CZ_DEVERR_SYM;
      sym = 0;  // keep walking with the warp, result is discarded
      sym_bad = true;
    }
    double acc = 0.0;
    uint32_t lo = 0, hi = 0;
    const int n_walk = (int)sym < V ? (int)sym + 1 : V;  // vocab part of the prefix
    cdf_walk<!kCache>(p, ld, n_walk, [&](int v, float x) {
      acc = __dadd_rn(acc, pdf_vocab(x));
      if ((uint32_t)v + 1 == sym) lo = quant(acc);
      if ((uint32_t)v == sym) hi = quant(acc);
      return (uint32_t)v < sym;
    });
    if (MODE == CZ_CDF_RWKV_LITERALS && (int)sym >= V) {  // literal symbols follow the vocab
      for (uint32_t v = (uint32_t)V; v <= sym; v++) {
        acc = __dadd_rn(acc, pdf_literal);
        if (v + 1 == sym) lo = quant(acc);
        if (v == sym) hi = quant(acc);
      }
    }
    if (hi < lo) hi = lo;                             // non-decreasing clamp (src/main.rs:818)
    if ((int)sym == n_sym - 1) hi = CZ_AC_CDF_TOTAL;  // cdf[n] = total (src/main.rs:822)
    lo_out = sym_bad ? 0u : lo;
    hi_out = sym_bad ? 0u : hi;
    return;
  }

  if (OP == OP_SEARCH) {
    const uint32_t value = arg;
    double acc = 0.0;
    uint32_t prev = 0, found_sym = (uint32_t)(n_sym - 1), lo = 0, hi = CZ_AC_CDF_TOTAL;
    bool done = false;
    auto visit = [&](int v, double pr) {
      acc = __dadd_rn(acc, pr);
      uint32_t cur = quant(acc);
      if (cur < prev) cur = prev;
      if (v == n_sym - 1) cur = CZ_AC_CDF_TOTAL;
      if (value < cur) {
        found_sym = (uint32_t)v;
        lo = prev;
        hi = cur;
        done = true;
      }
      prev = cur;
    };
    cdf_walk<!kCache>(p, ld, V, [&](int v, float x) {
      visit(v, pdf_vocab(x));
      return !done;
    });
    if (MODE == CZ_CDF_RWKV_LITERALS)
      for (int v = V; v < n_sym && !done; v++) visit(v, pdf_literal);
    sym_out = found_sym;
    lo_out = lo;
    hi_out = hi;
  }
}

}  // namespace czk
