// Round-2 CDF arithmetic: the same values as cdf_device.cuh, bit for bit, in far fewer issue slots.
//
// What bounded the round-1 kernel (profiles/ncu_summary_r01g.md: 33 instructions per logit, 58% issue, 0.32 of HBM) was not the
// ten FP64 operations of the glibc expf but what surrounds them:
//   * three F2F conversions per logit (f32 -> f64 of the argument, f64 -> f32 -> f64 of the result).  Conversions to / from 64-bit
//     types run at a quarter of the FP64 rate, so they cost more pipe time than the arithmetic.  Here the argument is widened with
//     one integer multiply-add ((u64)bits * 2^29 + bias: exact for a normal f32) and the result is rounded to the f32 grid
//     (round-to-nearest-even at mantissa bit 29) by integer adds on the f64 bit pattern -- valid while the result is a normal f32,
//     i.e. for max - logit <= 87; anything else (tiny results, -inf logits, NaN) takes the original conversion path, decided once
//     per group of rows.  cz_test_expf_exhaustive checks fast == original for every one of the 2^31 + NaN argument patterns.
//   * an IEEE division per element in every pass after the sum (p = e / S; the RWKV alphabet divides three times).  The divisor is
//     a per-column constant, so its correctly rounded reciprocal y = RN(1 / b) is computed once and each quotient costs five
//     FMA-pipe operations:  q0 = RN(a y);  r0 = RN(a - b q0);  q1 = RN(q0 + r0 y);  r1 = a - b q1 (exact);  q = RN(q1 + r1 y).
//     q1 is a faithful quotient (error < 1 ulp), and Markstein's theorem (Handbook of Floating-Point Arithmetic, thm 4.10: y within
//     1/2 ulp of 1/b, q1 faithful  =>  RN(q1 + r1 y) = RN(a / b)) makes q the correctly rounded quotient, i.e. __ddiv_rn(a, b).
//     cz_test_div_random compares the two on random operand pairs of the shapes that occur here (2^34 in the test suite).
//   * the encode-side prefix walk stops at the coded symbol, but with a thread per column a warp walks until its LAST lane stops:
//     with real token ids (mean id / V = 0.1, heavy tail) some lane of 32 nearly always needs most of the vocabulary.  The prefix
//     kernel is therefore warp-per-column (cdf_bounds_warp_kernel: the lanes evaluate 32 consecutive pdf entries, only the in-order
//     accumulation is serial), and it reads the e_v the stats pass left for it in a compact per-column cache instead of the
//     vocab-major logits (cdf_kernels.cu, "e-cache").
// The decode-side search (cdf_search_warp_n, below) uses the same fast paths.
#pragma once
#include "cdf_device.cuh"

namespace czk {

// 64-bit [entry][lane] copy of the exp2 table: one conflict-free LDS.64 per lookup (a half-warp's 16 lanes hit 16 distinct
// 8-byte bank pairs)
__device__ __forceinline__ void exp_tab64_init(uint64_t *s_tab) {
  for (int i = threadIdx.x; i < 32 * 32; i += blockDim.x) s_tab[i] = c_exp2f_tab[i >> 5];
  __syncthreads();
}

constexpr float CZ_EXP_FAST_MAX = 87.0f;  // e^-87 = 1.6e-38 > 2^-126: the result is a normal f32

// (double)expf(-a) for 0 <= a <= CZ_EXP_FAST_MAX (a = max - logit), identical to (double)cz_expf(-a): the operation sequence of
// cz_expf on the negated constant (RN is sign-symmetric), with the conversions done in integer arithmetic.
// tab_lane = table base + lane.
__device__ __forceinline__ double cz_exp_neg_fast(float a, const uint64_t *__restrict__ tab_lane) {
  const double ninv = -(0x1.71547652b82fep+0 * 32);
  const double shift = 0x1.8p+52;
  const double c0 = 0x1.c6af84b912394p-5 / 32 / 32 / 32;
  const double c1 = 0x1.ebfce50fac4f3p-3 / 32 / 32;
  const double c2 = 0x1.62e42ff0c52d6p-1 / 32;
  // f32 -> f64 of a normal non-negative float: exponent rebias 0x380 << 52, mantissa << 29.  For a = 0 or a subnormal this yields
  // a value below 2^-126 instead: harmless, both give expf = 1.0f exactly (|x| < 2^-25 rounds to 1).
  const uint64_t w = (uint64_t)__float_as_uint(a) * 0x20000000ull + 0x3800000000000000ull;
  const double ad = __longlong_as_double((long long)w);
  const double z = __dmul_rn(ninv, ad);
  double kd = __dadd_rn(z, shift);
  const uint32_t ki = (uint32_t)__double2loint(kd);
  kd = __dsub_rn(kd, shift);
  const double r = __fma_rn(ninv, ad, -kd);
  // (explicit shared-window address: lane slot + entry * 256 bytes is one LOP3 + one IMAD; through the generic pointer the compiler
  // rebuilds the lane part of the index for every lookup)
  uint64_t t;
  asm("ld.shared.u64 %0, [%1];" : "=l"(t) : "r"((uint32_t)__cvta_generic_to_shared(tab_lane) + ((ki & 31u) << 8)));
  const double s = __hiloint2double((int)((uint32_t)(t >> 32) + (ki << 15)), (int)(uint32_t)t);  // t += ki << 47
  const double p = __fma_rn(c0, r, c1);
  const double r2 = __dmul_rn(r, r);
  double y = __fma_rn(c2, r, 1.0);
  y = __fma_rn(p, r2, y);
  y = __dmul_rn(y, s);
  // RN-even to 24 significant bits: add half an f32 ulp minus one, plus the parity of the bit that stays; clear the 29 dropped bits
  uint64_t yb = (uint64_t)__double_as_longlong(y);
  yb += 0x0FFFFFFFull + ((yb >> 29) & 1ull);
  yb &= ~0x1FFFFFFFull;
  return __longlong_as_double((long long)yb);
}

// the f32 bit pattern of a double that lies on the normal-f32 grid (what cz_exp_neg_fast returns)
__device__ __forceinline__ float cz_f32_of_gridded(double d) {
  const uint32_t hi = (uint32_t)__double2hiint(d), lo = (uint32_t)__double2loint(d);
  return __uint_as_float(__funnelshift_l(lo, hi - 0x38000000u, 3));
}

// exact f32 -> f64 for values that only matter when they are >= 2^-126 (see above): one IMAD.WIDE instead of an F2F
__device__ __forceinline__ double cz_widen_pos(float e) {
  return __longlong_as_double((long long)((uint64_t)__float_as_uint(e) * 0x20000000ull + 0x3800000000000000ull));
}

// (cz_div_rcp / cz_div_rcp_ok: cdf_device.cuh -- the decode-side search uses them too)

// ---- vectorised full-column walk: NCOL adjacent columns per thread ------------------------------------------------------------
template <int NCOL>
struct CdfVec;
template <>
struct CdfVec<1> {
  using T = float;
  static __device__ __forceinline__ void unpack(const T &t, float (&x)[1]) { x[0] = t; }
};
template <>
struct CdfVec<2> {
  using T = float2;
  static __device__ __forceinline__ void unpack(const T &t, float (&x)[2]) {
    x[0] = t.x;
    x[1] = t.y;
  }
};
template <>
struct CdfVec<4> {
  using T = float4;
  static __device__ __forceinline__ void unpack(const T &t, float (&x)[4]) {
    x[0] = t.x;
    x[1] = t.y;
    x[2] = t.z;
    x[3] = t.w;
  }
};

// Calls f(v0, rows, cnt) for consecutive groups of up to GRP rows (cnt valid) of the NCOL columns starting at p, in ascending
// row order, with the next group's loads in flight and an L2 prefetch CDF_PF rows ahead (cdf_walk's pipelining).  NC: read-only path.
template <int NCOL, int GRP, bool NC, class F>
__device__ __forceinline__ void cdf_walk_groups(const float *p, size_t ld, int n, F f) {
  using T = typename CdfVec<NCOL>::T;
  auto ldv = [&](size_t row) -> T {
    const T *q = reinterpret_cast<const T *>(p + row * ld);
    return NC ? __ldg(q) : *q;
  };
  T cur[GRP], nxt[GRP];
  const T zero = T();
#pragma unroll
  for (int k = 0; k < GRP; k++) cur[k] = k < n ? ldv((size_t)k) : zero;
  int v0 = 0;
  for (; v0 + CDF_PF + GRP <= n; v0 += GRP) {
#pragma unroll
    for (int k = 0; k < GRP; k++) {
      nxt[k] = ldv((size_t)(v0 + GRP + k));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p + (size_t)(v0 + CDF_PF + k) * ld));
    }
    f(v0, cur, GRP);
#pragma unroll
    for (int k = 0; k < GRP; k++) cur[k] = nxt[k];
  }
  for (; v0 < n; v0 += GRP) {
#pragma unroll
    for (int k = 0; k < GRP; k++) {
      const int v = v0 + GRP + k;
      nxt[k] = v < n ? ldv((size_t)v) : zero;
    }
    f(v0, cur, n - v0 < GRP ? n - v0 : GRP);
#pragma unroll
    for (int k = 0; k < GRP; k++) cur[k] = nxt[k];
  }
}

// per-column results of the full passes, consumed by the prefix / XE kernels
struct __align__(16) CdfStats {
  double S;      // sum_i (f64)expf(l_i - max)                                        (src/main.rs:789-793)
  double norm;   // sum_i max(e_i / S, 2^-29)          (softmax_pdf_floor, :763-764)  -- floored alphabets and XE only, else 1
  double sum2;   // combined_pdf_with_literals' second normaliser (:773-779)           -- RWKV alphabet only, else 1
  float mx;      // max_i l_i
  int pad;
};

// (double)expf(-a) for a group of values: integer-conversion fast path when every a <= CZ_EXP_FAST_MAX, otherwise the original
// conversion path for the whole group (tiny results, -inf logits, NaN).  ef (optional) receives the f32 values.
template <int N, bool WANT_F32>
__device__ __forceinline__ void exp_group(const float (&a)[N], const ExpTab64 &tab, double (&d)[N], float (&ef)[N]) {
  // The fast path is evaluated unconditionally (garbage, but harmless, for arguments it does not cover) and a group that holds
  // such an argument is redone on the conversion path afterwards: the common case stays one straight-line block, which lets the
  // compiler interleave it with the caller's sequential f64 chains.
  bool ok = true;
#pragma unroll
  for (int i = 0; i < N; i++) {
    ok = ok && (a[i] <= CZ_EXP_FAST_MAX);
    d[i] = cz_exp_neg_fast(a[i], tab.t);
    if (WANT_F32) ef[i] = cz_f32_of_gridded(d[i]);
  }
  if (!ok) {
#pragma unroll
    for (int i = 0; i < N; i++) {
      const float e = cz_expf(-a[i], tab);
      d[i] = (double)e;
      if (WANT_F32) ef[i] = e;
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Warp-level search for the stepwise decoder: one warp walks NC columns (streams) at once.  With only hundreds of columns per
// step a thread-per-column walk is a ~10^5-deep dependent chain per thread with nothing to overlap.  Here the 32 lanes evaluate
// expf / the pdf for 32 consecutive vocab entries in parallel and only the order-dependent f64 accumulation is serial (every lane
// performs it redundantly on values exchanged through a shared-memory line, so all lanes hold the same S / acc and branches stay
// warp-uniform).  Same operations in the same order per column as cdf_col => bit-identical results.
//
// What a step costs is the latency of one warp's instruction stream (one or two warps per scheduler), so the loop is built for
// the in-order issue of a single warp (ncu, profiles/ncu_summary_r02.md: the first version took 1,240 cycles per group of 32 rows
// against the 262 of its 32 dependent adds -- 38% `wait`, 35% `long_scoreboard`, issue 16%):
//   * the columns' rows arrive through a per-warp shared-memory ring filled by cp.async four groups ahead: no register ring (whose
//     rotating moves wait for the newest load), and a decode batch's logits (V x streams x 4 bytes) come from DRAM;
//   * the next group's pdf entries are evaluated by a BRANCH-FREE fast path placed in the same basic block as the current group's
//     unconditional adds, so the scheduler interleaves the dependent chains; whether a lane's argument was outside the fast
//     path's domain is looked at after the adds, and only then is the value redone on the general path;
//   * NC = 2 columns per warp: their two add chains are independent, so each fills the other's 8-cycle DADD latency;
//   * the search adds whole groups and compares once per group (acc never decreases); the group that holds a column's crossing is
//     re-walked element by element.
// p[c]: column base (vocab-major, element v at p[c][v*ld]).  Must be called by a full warp; columns may repeat (a warp with one
// live stream passes it twice and ignores the second result).
// xch: NC * 128 doubles (NC KB) of shared memory private to the calling warp, 16-byte aligned: exchange lines + the row rings.
template <int MODE, int NC>
__device__ __forceinline__ void cdf_search_warp_n(const float *const (&p)[NC], size_t ld, int V, const uint32_t (&value)[NC],
                                                  const float (&mx)[NC], const ExpTab64 &tab, uint32_t (&sym_out)[NC],
                                                  uint32_t (&lo_out)[NC], uint32_t (&hi_out)[NC], int &errbits, double *xch) {
  // (No in-place caching of expf here, unlike cdf_col: the stepwise RWKV decoder keeps a stream's logits column across steps while
  // it decodes literal bytes, so the column must stay intact.)
  const int lane = threadIdx.x & 31;
  const int n_sym = MODE == CZ_CDF_RWKV_LITERALS ? V + 256 : V;
  const int n_full = V / 32, n_grp = (V + 31) / 32;
  constexpr int SR_DEPTH = 4;  // groups in flight (power of two)
  float *ring = reinterpret_cast<float *>(xch + NC * 64);
  const uint32_t ring_u32 = (uint32_t)__cvta_generic_to_shared(ring) + (uint32_t)lane * 4u;
  auto line_of = [&](int c, int buf) -> double * { return xch + (c * 2 + buf) * 32; };
  auto issue = [&](int g) {  // this lane's row of group g of every column -> ring slot g % SR_DEPTH; one commit group per call
    const int v = g * 32 + lane;
    if (v < V) {
#pragma unroll
      for (int c = 0; c < NC; c++)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(ring_u32 + (uint32_t)((c * SR_DEPTH + (g & (SR_DEPTH - 1))) * 128)),
                     "l"(p[c] + (size_t)v * ld)
                     : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  auto take = [&](int g, float (&x)[NC]) {  // (after issue(g + SR_DEPTH - 1): at most SR_DEPTH - 1 younger groups may still be pending)
    asm volatile("cp.async.wait_group %0;" ::"n"(SR_DEPTH - 1) : "memory");
    const int v = g * 32 + lane;
#pragma unroll
    for (int c = 0; c < NC; c++) x[c] = v < V ? ring[(c * SR_DEPTH + (g & (SR_DEPTH - 1))) * 32 + lane] : mx[c];  // rows beyond V are never added
  };
  auto drain = [&]() { asm volatile("cp.async.wait_all;" ::: "memory"); };
  // One in-order pass per column: out[c] = ((0 + f(c, x_0)) + f(c, x_1)) + ...   ffast(c, x, ok): branch-free, its value is only
  // used if ok; fslow(c, x): the general path, same value wherever ffast is ok.
  auto seq_sum = [&](auto ffast, auto fslow, double (&out)[NC]) {
    double acc[NC], q[NC];
    float xn[NC], x2[NC];
#pragma unroll
    for (int k = 0; k < SR_DEPTH; k++) issue(k);
    take(0, xn);
#pragma unroll
    for (int c = 0; c < NC; c++) {
      acc[c] = 0.0;
      q[c] = fslow(c, xn[c]);
    }
    issue(SR_DEPTH);
    take(1, xn);  // group g + 1's rows are read out of the ring one iteration before they are used
    for (int g = 0; g < n_full; g++) {
      issue(g + 1 + SR_DEPTH);
      take(g + 2, x2);
#pragma unroll
      for (int c = 0; c < NC; c++) line_of(c, g & 1)[lane] = q[c];
      __syncwarp();
      bool ok[NC];
      double qn[NC];
#pragma unroll
      for (int c = 0; c < NC; c++) qn[c] = ffast(c, xn[c], ok[c]);
#pragma unroll
      for (int k = 0; k < 32; k += 2) {
#pragma unroll
        for (int c = 0; c < NC; c++) {
          const double2 v = *reinterpret_cast<const double2 *>(line_of(c, g & 1) + k);
          acc[c] = __dadd_rn(acc[c], v.x);
          acc[c] = __dadd_rn(acc[c], v.y);
        }
      }
#pragma unroll
      for (int c = 0; c < NC; c++) {
        if (!ok[c]) qn[c] = fslow(c, xn[c]);
        q[c] = qn[c];
        xn[c] = x2[c];
      }
    }
    if (n_full < n_grp) {  // the ragged last group
#pragma unroll
      for (int c = 0; c < NC; c++) line_of(c, n_full & 1)[lane] = q[c];
      __syncwarp();
      const int cnt = V - n_full * 32;
      for (int k = 0; k < cnt; k++) {
#pragma unroll
        for (int c = 0; c < NC; c++) acc[c] = __dadd_rn(acc[c], line_of(c, n_full & 1)[k]);
      }
    }
    __syncwarp();
    drain();
#pragma unroll
    for (int c = 0; c < NC; c++) out[c] = acc[c];
  };
  // (double)expf(x - max): integer-conversion fast path for max - x <= 87 (cz_exp_neg_fast), else the original conversion path
  auto ex_fast = [&](int c, float x, bool &ok) -> double {
    const float a = __fsub_rn(mx[c], x);
    ok = a <= CZ_EXP_FAST_MAX;  // (false for NaN)
    return cz_exp_neg_fast(a, tab.t);
  };
  auto ex_slow = [&](int c, float x) -> double { return (double)cz_expf(__fsub_rn(x, mx[c]), tab); };
  double S[NC], norm[NC], sum2[NC], yS[NC], yN[NC], y2[NC];
  seq_sum(ex_fast, ex_slow, S);
  const double scale = 1.0 - 256.0 * CZ_P_FLOOR;
  // every division by a per-column constant: correctly rounded quotient from the constant's reciprocal (cz_div_rcp, proof above)
  // when the constant is in the proven range, else the IEEE division (the same value) -- decided once, for all NC columns, outside
  // the loops
  bool okS = true, any_uniform = false;
#pragma unroll
  for (int c = 0; c < NC; c++) {
    if (!(S[c] == S[c])) errbits |= CZ_DEVERR_NAN;
    okS = okS && cz_div_rcp_ok(S[c]);
    yS[c] = __drcp_rn(S[c]);
    norm[c] = 1.0;
    sum2[c] = 1.0;
    any_uniform = any_uniform || (MODE == CZ_CDF_SMOLLM && S[c] <= 0.0);  // src/main.rs:794-798
  }
  if (MODE != CZ_CDF_SMOLLM) {  // softmax_pdf_floor's normaliser (src/main.rs:763-764): the RWKV and the floored SmolLM alphabet
    if (okS) {
      auto g = [&](int c, double e) { return fmax(cz_div_rcp(e, S[c], yS[c]), CZ_P_FLOOR); };
      seq_sum([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); }, norm);
    } else {
      auto g = [&](int c, double e) { return fmax(__ddiv_rn(e, S[c]), CZ_P_FLOOR); };
      seq_sum([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); }, norm);
    }
  }
  if (MODE == CZ_CDF_RWKV_LITERALS) {
    bool okN = okS;
#pragma unroll
    for (int c = 0; c < NC; c++) {
      okN = okN && cz_div_rcp_ok(norm[c]);
      yN[c] = __drcp_rn(norm[c]);
    }
    if (okN) {
      auto g = [&](int c, double e) { return __dmul_rn(cz_div_rcp(fmax(cz_div_rcp(e, S[c], yS[c]), CZ_P_FLOOR), norm[c], yN[c]), scale); };
      seq_sum([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); }, sum2);
    } else {
      auto g = [&](int c, double e) { return __dmul_rn(__ddiv_rn(fmax(__ddiv_rn(e, S[c]), CZ_P_FLOOR), norm[c]), scale); };
      seq_sum([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); }, sum2);
    }
#pragma unroll
    for (int c = 0; c < NC; c++)
      for (int j = 0; j < 256; j++) sum2[c] = __dadd_rn(sum2[c], CZ_P_FLOOR);
  }
  bool fastd = okS;
#pragma unroll
  for (int c = 0; c < NC; c++) {
    fastd = fastd && cz_div_rcp_ok(norm[c]) && cz_div_rcp_ok(sum2[c]);
    yN[c] = __drcp_rn(norm[c]);
    y2[c] = __drcp_rn(sum2[c]);
  }
  const double uni = 1.0 / (double)V;
  // Search: per column the first v with value < cdf[v + 1].  cdf[v + 1] = floor(acc_v * 2^30) (clamped, made non-decreasing --
  // which a non-decreasing acc already is), so  value < cdf[v + 1]  <=>  acc_v * 2^30 >= value + 1  <=>  acc_v >= (value + 1) * 2^-30:
  // the scaling by a power of two is exact on both sides, so the test is ONE f64 compare against a constant instead of a
  // quantisation (multiply, clamp, convert) per element; the two bounds are quantised once, from acc_{v-1} and acc_v.
  double thr[NC], acc[NC], acc_prev[NC];
  uint32_t found[NC];
  bool done[NC];
#pragma unroll
  for (int c = 0; c < NC; c++) {
    thr[c] = __dmul_rn((double)value[c] + 1.0, 0x1p-30);
    acc[c] = 0.0;
    acc_prev[c] = 0.0;
    found[c] = (uint32_t)(n_sym - 1);
    done[c] = false;
  }
  auto all_done = [&]() {
    bool d = true;
#pragma unroll
    for (int c = 0; c < NC; c++) d = d && done[c];
    return d;
  };
  // re-walks one group of `cnt` values of column c element by element from acc[c] (the crossing, or the alphabet's end, is in it)
  auto scan_group = [&](int c, const double *line, int v0, int cnt) {
    for (int k = 0; k < cnt; k++) {
      const double a2 = __dadd_rn(acc[c], line[k]);
      const int v = v0 + k;
      if (a2 >= thr[c] || v == n_sym - 1) {
        found[c] = (uint32_t)v;
        acc_prev[c] = acc[c];
        acc[c] = a2;
        done[c] = true;
        break;
      }
      acc[c] = a2;
    }
  };
  // walks the vocabulary with pdf = pfast / pslow (same contract as seq_sum's pair) until every column has its crossing
  auto search = [&](auto pfast, auto pslow) {
    double q[NC];
    float xn[NC], x2[NC];
#pragma unroll
    for (int k = 0; k < SR_DEPTH; k++) issue(k);
    take(0, xn);
#pragma unroll
    for (int c = 0; c < NC; c++) q[c] = pslow(c, xn[c]);
    issue(SR_DEPTH);
    take(1, xn);
    int g = 0;
    for (; g < n_full && !all_done(); g++) {
      issue(g + 1 + SR_DEPTH);
      take(g + 2, x2);
#pragma unroll
      for (int c = 0; c < NC; c++) line_of(c, g & 1)[lane] = q[c];
      __syncwarp();
      bool ok[NC];
      double qn[NC], a[NC];
#pragma unroll
      for (int c = 0; c < NC; c++) {
        qn[c] = pfast(c, xn[c], ok[c]);
        a[c] = acc[c];
      }
#pragma unroll
      for (int k = 0; k < 32; k += 2) {
#pragma unroll
        for (int c = 0; c < NC; c++) {
          const double2 v = *reinterpret_cast<const double2 *>(line_of(c, g & 1) + k);
          a[c] = __dadd_rn(a[c], v.x);
          a[c] = __dadd_rn(a[c], v.y);
        }
      }
#pragma unroll
      for (int c = 0; c < NC; c++) {
        if (!ok[c]) qn[c] = pslow(c, xn[c]);
        q[c] = qn[c];
        xn[c] = x2[c];
        if (!done[c]) {  // (warp-uniform)
          if (a[c] >= thr[c] || g * 32 + 32 >= n_sym) scan_group(c, line_of(c, g & 1), g * 32, 32);
          else acc[c] = a[c];
        }
      }
    }
    if (n_full < n_grp && !all_done()) {  // the ragged last group of the vocabulary (only reached with g == n_full)
#pragma unroll
      for (int c = 0; c < NC; c++) line_of(c, n_full & 1)[lane] = q[c];
      __syncwarp();
#pragma unroll
      for (int c = 0; c < NC; c++)
        if (!done[c]) scan_group(c, line_of(c, n_full & 1), n_full * 32, V - n_full * 32);
    }
    __syncwarp();
    drain();
  };
  if (any_uniform || !fastd) {
    // degenerate columns (S <= 0: the reference's uniform pdf; constants outside the reciprocal's proven range): everything on the
    // general path, per-column branches and IEEE divisions
    auto g = [&](int c, double e) -> double {
      if (MODE == CZ_CDF_RWKV_LITERALS) {
        const double q = __dmul_rn(__ddiv_rn(fmax(__ddiv_rn(e, S[c]), CZ_P_FLOOR), norm[c]), scale);
        return sum2[c] > 0.0 ? __ddiv_rn(q, sum2[c]) : q;
      }
      if (MODE == CZ_CDF_SMOLLM_FLOOR) return __ddiv_rn(fmax(__ddiv_rn(e, S[c]), CZ_P_FLOOR), norm[c]);
      return S[c] <= 0.0 ? uni : __ddiv_rn(e, S[c]);
    };
    search([&](int, float, bool &ok) { ok = false; return 0.0; }, [&](int c, float x) { return g(c, ex_slow(c, x)); });
  } else if (MODE == CZ_CDF_RWKV_LITERALS) {
    // (fastd => sum2 is in cz_div_rcp's range, in particular > 0: the reference's `sum2 > 0` case, the block stays branch-free)
    auto g = [&](int c, double e) {
      return cz_div_rcp(__dmul_rn(cz_div_rcp(fmax(cz_div_rcp(e, S[c], yS[c]), CZ_P_FLOOR), norm[c], yN[c]), scale), sum2[c], y2[c]);
    };
    search([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); });
  } else if (MODE == CZ_CDF_SMOLLM_FLOOR) {
    auto g = [&](int c, double e) { return cz_div_rcp(fmax(cz_div_rcp(e, S[c], yS[c]), CZ_P_FLOOR), norm[c], yN[c]); };
    search([&](int c, float x, bool &ok) { return g(c, ex_fast(c, x, ok)); }, [&](int c, float x) { return g(c, ex_slow(c, x)); });
  } else {
    search([&](int c, float x, bool &ok) { return cz_div_rcp(ex_fast(c, x, ok), S[c], yS[c]); },
           [&](int c, float x) { return cz_div_rcp(ex_slow(c, x), S[c], yS[c]); });
  }
#pragma unroll
  for (int c = 0; c < NC; c++) {
    if (MODE == CZ_CDF_RWKV_LITERALS && !done[c]) {  // literal symbols follow the vocabulary
      const double pl = sum2[c] > 0.0 ? __ddiv_rn(CZ_P_FLOOR, sum2[c]) : CZ_P_FLOOR;
      for (int v = V; v < n_sym; v++) {
        const double a2 = __dadd_rn(acc[c], pl);
        if (a2 >= thr[c] || v == n_sym - 1) {
          found[c] = (uint32_t)v;
          acc_prev[c] = acc[c];
          acc[c] = a2;
          done[c] = true;
          break;
        }
        acc[c] = a2;
      }
    }
    // (done[c] is always true here: the last symbol ends the search)
    uint32_t lo = found[c] == 0 ? 0u : quant(acc_prev[c]);
    uint32_t hi = quant(acc[c]);
    if (hi < lo) hi = lo;
    if ((int)found[c] == n_sym - 1) hi = CZ_AC_CDF_TOTAL;
    sym_out[c] = found[c];
    lo_out[c] = lo;
    hi_out[c] = hi;
  }
}

}  // namespace czk
