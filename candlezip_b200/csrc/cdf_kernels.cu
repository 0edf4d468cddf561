// K1 / K9: logits -> quantised integer CDF bounds, CDF search, cross-entropy bits.
//
// Replaces src/main.rs:784-824 (softmax_pdf + quantize_pdf_to_cdf), 758-782 (softmax_pdf_floor,
// combined_pdf_with_literals), 2294-2326 (encode-side use), 2622-2625 (decode-side search), 1743-1749 /
// 1776-1784 (XE accumulation).  The reference's arithmetic is ORDER-DEPENDENT f64 (sequential sum over the
// vocab, sequential prefix), so bit-exact parity forbids tree reductions: one thread owns one column (one
// stream / one teacher-forced position) and walks the vocab in ascending order.  Parallelism comes from the
// columns (all positions of all chunks are independent on the encode side).  Logits are VOCAB-MAJOR
// [V][ld] so that the 32 columns of a warp read one coalesced 128-byte line per vocab entry.
//
// expf: identical operation sequence to glibc 2.39 x86_64 expf (the FMA ifunc variant), which is what Rust's
// f32::exp lowers to on Linux; every mul/add/fma is an explicit round-to-nearest intrinsic so nvcc cannot
// re-contract.  Algorithmic bytes = 4*V per column (one read).  Encode (OP_BOUNDS / OP_XE): the max comes from the LM-head
// GEMM's epilogue, cdf_stats_tma_kernel reads the column once per pass (one pass for SmolLM coding) and leaves the few e_v the
// prefix walk needs in a compact cache, cdf_bounds_warp_kernel walks that cache; cdf_stats_kernel does the same passes by direct
// loads for batches the tensor map cannot describe (ld % 4 != 0, an unaligned base) or too small to fill the machine.
// Decode (OP_SEARCH): cdf_search_warp_n (cdf_fast.cuh), a warp per stream.
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "cdf_fast.cuh"
#include "tc_ptx.cuh"

namespace czk {

// =================================================================================================================
// Round-2 encode-side kernels (OP_BOUNDS / OP_XE): full passes and the prefix walk are separate kernels.
// =================================================================================================================

// Full passes by direct loads, one thread per column, every column summed in ascending vocab order.  MODE / OP decide which passes run:
//   pass 1  S = sum (f64)expf(l - max)                      always            (RWKV alphabet: leaves e_v in the logit's slot)
//   pass 2  norm = sum max(e / S, 2^-29)                    RWKV alphabet, floored SmolLM alphabet, XE
//   pass 3  sum2 = sum RN(RN(max(e / S, 2^-29) / norm) (1 - 2^-21)) + 256 x 2^-29   RWKV alphabet
template <int MODE, int OP>
__global__ void __launch_bounds__(128) cdf_stats_kernel(float *__restrict__ logits, int V, size_t M, size_t ld, const int *__restrict__ colmax,
                                                        CdfStats *__restrict__ stats, int *__restrict__ err) {
  constexpr bool kLit = MODE == CZ_CDF_RWKV_LITERALS;
  constexpr bool kNorm = kLit || OP == OP_XE || MODE == CZ_CDF_SMOLLM_FLOOR;
  __shared__ uint64_t s_tab[32 * 32];
  exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  const size_t col = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= M) return;
  float *p = logits + col;
  float mx;
  if (colmax) {
    mx = colmax_decode(colmax[col]);
  } else {
    mx = __int_as_float(0xff800000);
    cdf_walk_groups<true>(p, ld, V, [&](int, const float(&x)[CDF_GRP], int cnt) {
#pragma unroll
      for (int k = 0; k < CDF_GRP; k++)
        if (k < cnt && x[k] > mx) mx = x[k];  // NaN-ignoring, like `if v > max` (src/main.rs:786-788)
    });
  }
  // ---- pass 1 ----
  double S = 0.0;
  cdf_walk_groups<!kLit>(p, ld, V, [&](int v0, const float(&x)[CDF_GRP], int cnt) {
    float a[CDF_GRP], ef[CDF_GRP];
    double d[CDF_GRP];
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) a[k] = __fsub_rn(mx, x[k]);  // = -(l - max), exactly
    exp_group<CDF_GRP, kLit>(a, tab, d, ef);
#pragma unroll
    for (int k = 0; k < CDF_GRP; k++) {
      if (k < cnt) {
        S = __dadd_rn(S, d[k]);
        if (kLit) p[(size_t)(v0 + k) * ld] = ef[k];  // cache e_v for the later passes
      }
    }
  });
  int errbits = 0;
  if (!(S == S)) errbits |= CZ_DEVERR_NAN;
  double norm = 1.0, sum2 = 1.0;
  if (kNorm) {
    // (spelled as a running AND on purpose: `const bool fast = cz_div_rcp_ok(S)` makes nvcc 12.9 build different code for the passes
    // below, e.g. 72 registers and 16 B of spill stores instead of 90 and none for XE and the floored alphabet)
    bool fast = true;
    fast = fast && cz_div_rcp_ok(S);
    const double yS = __drcp_rn(S);
    // e_v (as a double) of the rows of a group: the cached f32 (RWKV alphabet) or recomputed from the logit (SmolLM: floored / XE)
    auto e_of = [&](const float(&x)[CDF_GRP], double(&d)[CDF_GRP]) {
      float a[CDF_GRP], ef[CDF_GRP];
#pragma unroll
      for (int k = 0; k < CDF_GRP; k++) {
        if (kLit) d[k] = fast ? cz_widen_pos(x[k]) : (double)x[k];  // (values below 2^-126 are floored either way)
        else a[k] = __fsub_rn(mx, x[k]);
      }
      if (!kLit) exp_group<CDF_GRP, false>(a, tab, d, ef);
    };
    auto div_S = [&](double e) { return fast ? cz_div_rcp(e, S, yS) : __ddiv_rn(e, S); };
    // ---- pass 2 ----
    double acc = 0.0;
    cdf_walk_groups<!kLit>(p, ld, V, [&](int, const float(&x)[CDF_GRP], int cnt) {
      double d[CDF_GRP];
      e_of(x, d);
#pragma unroll
      for (int k = 0; k < CDF_GRP; k++)
        if (k < cnt) acc = __dadd_rn(acc, fmax(div_S(d[k]), CZ_P_FLOOR));
    });
    norm = acc;
    if (kLit) {
      // ---- pass 3 ----
      const double scale = 1.0 - 256.0 * CZ_P_FLOOR;
      const bool fastn = fast && cz_div_rcp_ok(norm);
      const double yN = __drcp_rn(norm);
      acc = 0.0;
      cdf_walk_groups<false>(p, ld, V, [&](int, const float(&x)[CDF_GRP], int cnt) {
        double d[CDF_GRP];
        e_of(x, d);
#pragma unroll
        for (int k = 0; k < CDF_GRP; k++)
          if (k < cnt) {
            const double q = fmax(div_S(d[k]), CZ_P_FLOOR);
            const double q2 = fastn ? cz_div_rcp(q, norm, yN) : __ddiv_rn(q, norm);
            acc = __dadd_rn(acc, __dmul_rn(q2, scale));
          }
      });
      for (int j = 0; j < 256; j++) acc = __dadd_rn(acc, CZ_P_FLOOR);
      sum2 = acc;
    }
  }
  CdfStats st;
  st.S = S;
  st.norm = norm;
  st.sum2 = sum2;
  st.mx = mx;
  st.pad = 0;
  stats[col] = st;
  if (errbits) atomicOr(err, errbits);
}


// ---------------------------------------------------------------------------------------------------------------------------------
// The e-cache: what the prefix walk needs, laid out for it.
// The prefix walk of column c adds e_v / S for v = 0 .. sym_c.  Reading those e_v (or the logits they come from) out of the
// vocab-major batch costs a whole 32-byte sector -- a 64-byte DRAM fetch -- per 4-byte value, because the walk lengths of adjacent
// columns have nothing to do with each other (ncu, profiles/ncu_summary_r02.md: 38 GB of DRAM reads per 131,072 columns against
// 2.6 GB of values used, the kernel sits at 72% of DRAM bandwidth).  The stats pass has every e_v in a register anyway, so the
// thread that owns column c also stores e_v (as the f64 it adds to S), for v <= sym_c only, CONTIGUOUSLY per column: groups of 8
// rows = 64 bytes, at a per-column offset from an exclusive scan of ceil((sym_c + 1) / 8).  The prefix walk then reads 256
// coalesced bytes per 32 rows and no longer evaluates expf.  Capacity is a fraction of the batch (real text: mean sym / V = 0.1);
// if a batch needs more, the flag stays 0 and the prefix walk reads the logits as before -- same values either way.
// ---------------------------------------------------------------------------------------------------------------------------------
constexpr int EC_GRP = 8;  // rows per cache group (64 bytes of f64)

__global__ void __launch_bounds__(1024) ecache_offsets_kernel(const uint32_t *__restrict__ syms, size_t M, int V, int n_sym,
                                                              uint32_t *__restrict__ eoff, unsigned long long cap_groups,
                                                              int *__restrict__ flag) {
  __shared__ unsigned long long s_warp[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t per = (M + 1023) / 1024, b = (size_t)tid * per, e = b + per < M ? b + per : M;
  auto groups = [&](size_t c) -> unsigned {
    const uint32_t sym = syms[c];
    if ((int)sym >= n_sym) return 0u;  // (reported by the prefix kernel)
    const int n = (int)sym < V ? (int)sym + 1 : V;
    return (unsigned)((n + EC_GRP - 1) / EC_GRP);
  };
  unsigned long long mine = 0;
  for (size_t c = b; c < e; c++) mine += groups(c);
  unsigned long long incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    unsigned long long w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  const unsigned long long total = s_warp[31];
  const bool fits = total <= cap_groups && total <= 0xffffffffull;
  if (tid == 0) {
    *flag = fits ? 1 : 0;
    eoff[M] = fits ? (uint32_t)total : 0u;
  }
  if (!fits) return;
  unsigned long long run = incl - mine + (warp ? s_warp[warp - 1] : 0ull);
  for (size_t c = b; c < e; c++) {
    eoff[c] = (uint32_t)run;
    run += groups(c);
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// Full passes with the logits STAGED THROUGH SHARED MEMORY BY TMA.  cdf_stats_kernel spends a third of its issue slots on getting
// the data: per logit one LDG, one L2 prefetch and four 64-bit address adds (rows are ld * 4 bytes apart, nothing folds into an
// immediate), and its top stall is the load scoreboard (ncu, profiles/ncu_summary_r02.md).  Here one elected thread per CTA streams
// [16 or 32 rows] x [256 columns] boxes (1 KB contiguous per row) into a shared-memory ring (StCfg) with cp.async.bulk.tensor;
// the 256 consumer threads (thread = column) read their values with immediate-offset LDS, so the per-logit cost is the arithmetic
// alone and the loads run arbitrarily far ahead of it.  Same values, same order per column: bit-identical to cdf_stats_kernel.
// Needs ld % 4 == 0 and a 16-byte aligned base (tensor-map strides); otherwise the launcher keeps cdf_stats_kernel.
// ---------------------------------------------------------------------------------------------------------------------------------
// Tile shape per alphabet, two CTAs per SM (measured on B200, scripts/cdf_bench.py, 131,072 columns, stats pass alone; three CTAs per SM
// cap the kernel at 75 registers and the compiler then re-materialises the polynomial's constants in every group of 8 rows):
//   SmolLM  16 rows x 4 stages x 3 CTAs 13.5 ms | 16 x 4 x 2 CTAs 12.0 | 16 x 6 x 2 12.0 | 32 x 3 x 2 11.6 | 32 x 2 x 2 11.9 | 8 x 8 x 2 12.7
//   RWKV    16 x 4 x 3 CTAs 53.1 ms | 16 x 4 x 2 50.5 | 16 x 6 x 2 50.2 | 32 x 3 x 2 52.1   (its first pass stores e_v in place, a barrier per pass)
constexpr int ST_COLS = 256;
template <int MODE>
struct StCfg {
  static constexpr int ROWS = MODE == CZ_CDF_RWKV_LITERALS ? 16 : 32;
  static constexpr int STAGES = MODE == CZ_CDF_RWKV_LITERALS ? 6 : 3;
  static constexpr int TILE_BYTES = ST_COLS * ROWS * 4;
  static constexpr int SMEM = STAGES * TILE_BYTES + 32 * 32 * 8 + 128;  // tiles | exp table | barriers
};

template <int MODE, int OP>
__global__ void __launch_bounds__(ST_COLS + 32, 2) cdf_stats_tma_kernel(const __grid_constant__ CUtensorMap tm, float *__restrict__ logits, int V,
                                                                       size_t M, size_t ld, const int *__restrict__ colmax,
                                                                       CdfStats *__restrict__ stats, int *__restrict__ err,
                                                                       const uint32_t *__restrict__ syms, const uint32_t *__restrict__ eoff,
                                                                       double *__restrict__ ecache, const int *__restrict__ eflag) {
  constexpr bool kLit = MODE == CZ_CDF_RWKV_LITERALS;
  constexpr bool kNorm = kLit || OP == OP_XE || MODE == CZ_CDF_SMOLLM_FLOOR;
  constexpr bool kSpill = OP == OP_BOUNDS;  // (ecache may still be null: no e-cache for this batch)
  constexpr int ST_ROWS = StCfg<MODE>::ROWS, ST_STAGES = StCfg<MODE>::STAGES, ST_TILE_BYTES = StCfg<MODE>::TILE_BYTES;
  extern __shared__ __align__(1024) uint8_t st_smem[];
  float *tiles = reinterpret_cast<float *>(st_smem);
  uint64_t *s_tab = reinterpret_cast<uint64_t *>(st_smem + ST_STAGES * ST_TILE_BYTES);
  uint64_t *bars = reinterpret_cast<uint64_t *>(st_smem + ST_STAGES * ST_TILE_BYTES + 32 * 32 * 8);
  const uint32_t full_bar = smem_u32(&bars[0]), empty_bar = smem_u32(&bars[ST_STAGES]);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int s2 = 0; s2 < ST_STAGES; s2++) {
      mbar_init(full_bar + 8 * s2, 1);
      mbar_init(empty_bar + 8 * s2, ST_COLS / 32);  // one arrival per consumer warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  exp_tab64_init(s_tab);  // (__syncthreads inside)
  const int n_tiles = (V + ST_ROWS - 1) / ST_ROWS;
  const bool need_max = colmax == nullptr;
  const int n_pass = (need_max ? 1 : 0) + 1 + (kNorm ? 1 : 0) + (kLit ? 1 : 0);
  const int c0 = blockIdx.x * ST_COLS;

  if (warp == ST_COLS / 32) {
    // ===================== producer warp: lane 0 issues the box loads =====================
    int it = 0;
    for (int pass = 0; pass < n_pass; pass++) {
      if (lane == 0) {
        if (pass == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&tm) : "memory");
        for (int t = 0; t < n_tiles; t++, it++) {
          const int st = it % ST_STAGES;
          mbar_wait(empty_bar + 8 * st, ((it / ST_STAGES) & 1) ^ 1);
          mbar_expect_tx(full_bar + 8 * st, ST_TILE_BYTES);
          tma_load_2d(smem_u32(tiles + (size_t)st * ST_COLS * ST_ROWS), &tm, full_bar + 8 * st, c0, t * ST_ROWS);
        }
      }
      __syncwarp();
      // the RWKV alphabet's first pass rewrites the batch in place (expf cache): its stores must be complete and visible to the
      // async proxy before the next pass's boxes are requested
      if (kLit && pass == (need_max ? 1 : 0)) asm volatile("bar.sync 1, %0;" ::"n"(ST_COLS + 32) : "memory");
    }
    return;
  }
  // ===================== consumers: thread = column =====================
  const ExpTab64 tab{s_tab + lane};
  const size_t col = (size_t)c0 + tid;
  const bool active = col < M;
  float mx = need_max ? __int_as_float(0xff800000) : (active ? colmax_decode(colmax[col]) : 0.f);
  int it = 0;
  // walks one pass: f(v0, x[8], cnt) per group of 8 rows, in ascending row order
  auto run_pass = [&](auto f) {
    for (int t = 0; t < n_tiles; t++, it++) {
      const int st = it % ST_STAGES;
      mbar_wait(full_bar + 8 * st, (it / ST_STAGES) & 1);
      const float *src = tiles + (size_t)st * ST_COLS * ST_ROWS + tid;
      if (t + 1 < n_tiles || V % ST_ROWS == 0) {
        // a full tile: compile-time groups of 8 rows (no per-element predicates), read 8 at a time (the registers of a whole tile
        // are better spent on keeping the polynomial's constants resident); the slot is handed back once its last group is read
#pragma unroll
        for (int g = 0; g < ST_ROWS / 8; g++) {
          float xg[8];
#pragma unroll
          for (int k = 0; k < 8; k++) xg[k] = src[(g * 8 + k) * ST_COLS];
          if (g == ST_ROWS / 8 - 1) {
            __syncwarp();
            if (lane == 0) mbar_arrive(empty_bar + 8 * st);
          }
          f(t * ST_ROWS + g * 8, xg, 8);
        }
        continue;
      }
      // the ragged last tile (rows beyond V are zero-filled by the tensor map; f ignores them)
      const int rows = V - t * ST_ROWS;
      for (int g = 0; g * 8 < rows; g++) {
        float xg[8];
#pragma unroll
        for (int k = 0; k < 8; k++) xg[k] = src[(g * 8 + k) * ST_COLS];
        const int cnt = rows - g * 8;
        f(t * ST_ROWS + g * 8, xg, cnt < 8 ? cnt : 8);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_bar + 8 * st);
    }
  };
  auto pass_barrier = [&]() {
    if (kLit) {
      asm volatile("fence.proxy.async.global;" ::: "memory");
      asm volatile("bar.sync 1, %0;" ::"n"(ST_COLS + 32) : "memory");
    }
  };
  if (need_max) {
    run_pass([&](int, const float(&x)[8], int cnt) {
#pragma unroll
      for (int k = 0; k < 8; k++)
        if (k < cnt && x[k] > mx) mx = x[k];  // NaN-ignoring, like `if v > max` (src/main.rs:786-788)
    });
  }
  // ---- pass 1: S ----
  // e-cache: this column's rows 0 .. sym go to ecache[eoff[col] * 8 ...] (see ecache_offsets_kernel)
  int n_spill = 0;
  double *edst = nullptr;
  if (kSpill && ecache != nullptr && active && *eflag != 0) {
    const uint32_t sym = syms[col];
    const int n_sym = kLit ? V + 256 : V;
    if ((int)sym < n_sym) n_spill = (int)sym < V ? (int)sym + 1 : V;
    edst = ecache + (size_t)eoff[col] * EC_GRP;
  }
  double S = 0.0;
  run_pass([&](int v0, const float(&x)[8], int cnt) {
    float a[8], ef[8];
    double d[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = __fsub_rn(mx, x[k]);  // = -(l - max), exactly
    exp_group<8, kLit>(a, tab, d, ef);
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (k < cnt) {
        S = __dadd_rn(S, d[k]);
        if (kLit && active) logits[(size_t)(v0 + k) * ld + col] = ef[k];  // cache e_v for the later passes
      }
    if (kSpill && v0 < n_spill) {  // (rows of the group beyond sym, or beyond V in the ragged tile, are never read)
      double2 *q = reinterpret_cast<double2 *>(edst + v0);
#pragma unroll
      for (int k = 0; k < 8; k += 2) q[k >> 1] = make_double2(d[k], d[k + 1]);
    }
  });
  int errbits = 0;
  if (active && !(S == S)) errbits |= CZ_DEVERR_NAN;
  double norm = 1.0, sum2 = 1.0;
  if (kNorm) {
    pass_barrier();
    // The reciprocal-based divisions are decided per WARP and outside the loops (the same values either way; a per-element
    // `fast ? ... : __ddiv_rn` left a branch and the IEEE division's code in every group: 14% `branch_resolving` and 6% instruction-
    // fetch stalls in the RWKV alphabet's passes, profiles/ncu_summary_r02.md).  Every consumer warp is whole, so the vote is safe.
    const bool fast = __all_sync(0xffffffffu, cz_div_rcp_ok(S));
    const double yS = __drcp_rn(S);
    // e_v of the 8 rows: the cached f32 (RWKV alphabet; WIDEN: exact integer widening, values below 2^-126 are floored either way)
    // or expf again (SmolLM's floored alphabet and XE pass)
    auto e_of = [&](const float(&x)[8], double(&d)[8], auto widen) {
      if (kLit) {
#pragma unroll
        for (int k = 0; k < 8; k++) d[k] = decltype(widen)::value ? cz_widen_pos(x[k]) : (double)x[k];
      } else {
        float a[8], ef[8];
#pragma unroll
        for (int k = 0; k < 8; k++) a[k] = __fsub_rn(mx, x[k]);
        exp_group<8, false>(a, tab, d, ef);
      }
    };
    // ---- pass 2: norm ----
    auto pass2 = [&](auto rcp) {
      double acc = 0.0;
      run_pass([&](int, const float(&x)[8], int cnt) {
        double d[8];
        e_of(x, d, rcp);
#pragma unroll
        for (int k = 0; k < 8; k++)
          if (k < cnt) acc = __dadd_rn(acc, fmax(decltype(rcp)::value ? cz_div_rcp(d[k], S, yS) : __ddiv_rn(d[k], S), CZ_P_FLOOR));
      });
      return acc;
    };
    norm = fast ? pass2(std::true_type{}) : pass2(std::false_type{});
    if (kLit) {
      // ---- pass 3: sum2 ----  (no stores since pass 1: no barrier needed, the producer may already be ahead)
      const double scale = 1.0 - 256.0 * CZ_P_FLOOR;
      const bool fastn = __all_sync(0xffffffffu, fast && cz_div_rcp_ok(norm));
      const double yN = __drcp_rn(norm);
      auto pass3 = [&](auto rcp) {
        double acc = 0.0;
        run_pass([&](int, const float(&x)[8], int cnt) {
          double d[8];
          e_of(x, d, rcp);
#pragma unroll
          for (int k = 0; k < 8; k++)
            if (k < cnt) {
              const double q = fmax(decltype(rcp)::value ? cz_div_rcp(d[k], S, yS) : __ddiv_rn(d[k], S), CZ_P_FLOOR);
              const double q2 = decltype(rcp)::value ? cz_div_rcp(q, norm, yN) : __ddiv_rn(q, norm);
              acc = __dadd_rn(acc, __dmul_rn(q2, scale));
            }
        });
        return acc;
      };
      double acc = fastn ? pass3(std::true_type{}) : pass3(std::false_type{});
      for (int j = 0; j < 256; j++) acc = __dadd_rn(acc, CZ_P_FLOOR);
      sum2 = acc;
    }
  }
  if (active) {
    CdfStats st;
    st.S = S;
    st.norm = norm;
    st.sum2 = sum2;
    st.mx = mx;
    st.pad = 0;
    stats[col] = st;
    if (errbits) atomicOr(err, errbits);
  }
}

// pdf entry of vocab element v from its logit (SmolLM) / cached e_v (RWKV alphabet): the same expressions as cdf_full_kernel's
template <int MODE, bool FLOORED>
struct PdfOf {
  double S, norm, sum2, yS, yN, y2, uni;
  bool fast, uniform, has2;
  __device__ __forceinline__ void init(const CdfStats &st, int V) {
    S = st.S;
    norm = st.norm;
    sum2 = st.sum2;
    fast = cz_div_rcp_ok(S) && cz_div_rcp_ok(norm) && cz_div_rcp_ok(sum2);
    yS = __drcp_rn(S);
    yN = __drcp_rn(norm);
    y2 = __drcp_rn(sum2);
    uniform = MODE == CZ_CDF_SMOLLM && !FLOORED && S <= 0.0;  // src/main.rs:794-798
    uni = 1.0 / (double)V;
    has2 = sum2 > 0.0;
  }
  __device__ __forceinline__ double dv(double a, double b, double y) const { return fast ? cz_div_rcp(a, b, y) : __ddiv_rn(a, b); }
  __device__ __forceinline__ double operator()(double e) const {
    if (MODE == CZ_CDF_RWKV_LITERALS) {
      double q = fmax(dv(e, S, yS), CZ_P_FLOOR);
      q = __dmul_rn(dv(q, norm, yN), 1.0 - 256.0 * CZ_P_FLOOR);
      return has2 ? dv(q, sum2, y2) : q;
    } else if (FLOORED) {
      return dv(fmax(dv(e, S, yS), CZ_P_FLOOR), norm, yN);
    } else {
      return uniform ? uni : dv(e, S, yS);
    }
  }
  // the same value with the division mode fixed at compile time (the walk decides once per column, outside its loop): F => every
  // constant is inside the reciprocal's proven range, in particular S > 0 (not the uniform case) and sum2 > 0
  template <bool F>
  __device__ __forceinline__ double get(double e) const {
    if (!F) {
      PdfOf t = *this;
      t.fast = false;
      return t(e);
    }
    if (MODE == CZ_CDF_RWKV_LITERALS)
      return cz_div_rcp(__dmul_rn(cz_div_rcp(fmax(cz_div_rcp(e, S, yS), CZ_P_FLOOR), norm, yN), 1.0 - 256.0 * CZ_P_FLOOR), sum2, y2);
    if (FLOORED) return cz_div_rcp(fmax(cz_div_rcp(e, S, yS), CZ_P_FLOOR), norm, yN);
    return cz_div_rcp(e, S, yS);
  }
  __device__ __forceinline__ double literal() const { return has2 ? __ddiv_rn(CZ_P_FLOOR, sum2) : CZ_P_FLOOR; }
};

// Prefix walk (encode): cdf[sym], cdf[sym + 1] of every column -- ONE WARP PER COLUMN.
//
// The walk is a strictly sequential f64 sum of sym + 1 terms, and symbols are heavy-tailed (mean id / V = 0.1 for real text, but
// one column in twenty needs more than half of the vocabulary).  With a thread per column a warp walks until its slowest lane is
// done, and even with the columns of a CTA sorted by symbol the kernel's duration was the latency of the lone warps left walking
// the longest columns (ncu, profiles/ncu_summary_r02.md: 1.2 warps per scheduler, 4,000 cycles per 8 rows, 9-13 ms per 131,072
// columns).  Here the 32 lanes of a warp evaluate the pdf entries of 32 consecutive vocab entries of ONE column in parallel (expf,
// divisions: the expensive part) and only the order-dependent accumulation is serial -- every lane performs it redundantly on the
// shared-memory line the values were exchanged through (cdf_search_warp's scheme), so all lanes hold the same acc and every branch
// is warp-uniform.  Columns are independent warps of very different lengths, thousands per SM over the kernel's life: the machine
// stays full until the end, and the longest column costs V / 32 short iterations.
// Same operations in the same order as cdf_full_kernel's prefix sum: bit-identical results.
// Columns are handed out one at a time from a global counter (persistent warps): a warp that finishes a short column takes the
// next one instead of idling until the longest column of its CTA is done.  (Reading the vocab-major logits this way was meant to
// share a row's 32-byte sector between the warps of adjacent columns through L1 / L2; ncu showed it does not -- the walks drift
// apart at once: 38 GB of DRAM reads per 131,072 columns for 2.6 GB used.  Hence the e-cache.)
// CACHED: the e_v come from the e-cache the stats pass filled (f64, contiguous per column: 256 coalesced bytes per 32 rows, no
// expf); the kernel is a no-op when the batch did not fit the cache (*eflag == 0).  !CACHED: from the vocab-major logits; a no-op
// when eflag is given and set.  The launcher issues both, exactly one of them works.
template <int MODE, bool CACHED>
__global__ void __launch_bounds__(256) cdf_bounds_warp_kernel(const float *__restrict__ logits, int V, size_t M, size_t ld,
                                                              const uint32_t *__restrict__ syms, const CdfStats *__restrict__ stats,
                                                              uint32_t *__restrict__ c_lo_out, uint32_t *__restrict__ c_hi_out,
                                                              int *__restrict__ err, unsigned int *__restrict__ work_counter,
                                                              const uint32_t *__restrict__ eoff, const double *__restrict__ ecache,
                                                              const int *__restrict__ eflag) {
  constexpr bool kLit = MODE == CZ_CDF_RWKV_LITERALS;
  constexpr int DEPTH = 4;  // groups of 32 rows whose loads are in flight ahead of the group being added
  __shared__ uint64_t s_tab[CACHED ? 32 : 32 * 32];
  __shared__ __align__(16) double s_xch[8 * 64];  // per warp: two 32-value exchange lines
  if (CACHED ? *eflag == 0 : (eflag != nullptr && *eflag != 0)) return;
  if (!CACHED) exp_tab64_init(s_tab);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const ExpTab64 tab{s_tab + (CACHED ? 0 : lane)};
  double *xch = s_xch + warp * 64;
  const int n_sym = kLit ? V + 256 : V;
  for (;;) {
    unsigned int c = 0;
    if (lane == 0) c = atomicAdd(work_counter, 1u);
    c = __shfl_sync(0xffffffffu, c, 0);
    if ((size_t)c >= M) return;
    const size_t col = c;
    const uint32_t sym = syms[col];
    if ((int)sym >= n_sym) {
      if (lane == 0) {
        atomicOr(err, CZ_DEVERR_SYM);
        c_lo_out[col] = 0u;
        c_hi_out[col] = 0u;
      }
      continue;
    }
    const CdfStats st = stats[col];
    PdfOf<MODE, MODE == CZ_CDF_SMOLLM_FLOOR> pdf;
    pdf.init(st, V);
    const float mx = st.mx;
    const float *p = logits + col;
    const int n = (int)sym < V ? (int)sym + 1 : V;  // vocab rows to add
    const int n_grp = (n + 31) >> 5;
    // the rows hold logits (SmolLM) or the e_v the stats kernel's first pass left there (RWKV alphabet)
    using X = typename std::conditional<CACHED, double, float>::type;
    const double *pe = CACHED ? ecache + (size_t)eoff[col] * EC_GRP : nullptr;
    auto ld_x = [&](int g) -> X {
      const int v = g * 32 + lane;
      if (CACHED) return v < n ? __ldg(pe + v) : 0.0;
      return v < n ? (kLit ? p[(size_t)v * ld] : __ldg(p + (size_t)v * ld)) : 0.f;
    };
    double acc = 0.0;
    uint32_t lo = 0, hi = 0;
    // the walk, with the division mode (reciprocal-based or IEEE: same values) fixed per column outside the loop
    auto walk = [&](auto fast_tag) {
      constexpr bool kFast = decltype(fast_tag)::value;
      auto q_of = [&](X x) -> double {
        double d;
        if (CACHED) {
          d = (double)x;
        } else if (kLit) {
          d = kFast ? cz_widen_pos(x) : (double)x;  // (values below 2^-126 are floored either way)
        } else {
          const float a1[1] = {__fsub_rn(mx, x)};
          double d1[1];
          float e1[1];
          exp_group<1, false>(a1, tab, d1, e1);
          d = d1[0];
        }
        return pdf.template get<kFast>(d);
      };
      X xr[DEPTH];
#pragma unroll
      for (int k = 0; k < DEPTH; k++) xr[k] = ld_x(k);
      for (int g = 0; g < n_grp; g++) {
        const X x = xr[0];
#pragma unroll
        for (int k = 0; k + 1 < DEPTH; k++) xr[k] = xr[k + 1];
        xr[DEPTH - 1] = ld_x(g + DEPTH);
        double *line = xch + (g & 1) * 32;
        line[lane] = q_of(x);
        __syncwarp();
        const int v0 = g * 32;
        if (v0 + 32 < (int)sym && v0 + 32 <= n) {  // (warp-uniform) a full group that ends before cdf[sym]'s last term: 32 plain adds
#pragma unroll
          for (int k = 0; k < 32; k += 2) {
            const double2 t = *reinterpret_cast<const double2 *>(line + k);
            acc = __dadd_rn(acc, t.x);
            acc = __dadd_rn(acc, t.y);
          }
        } else {  // at most the last two groups of a column
          const int cnt = n - v0 < 32 ? n - v0 : 32;
          for (int k = 0; k < cnt; k++) {
            acc = __dadd_rn(acc, line[k]);
            const uint32_t v = (uint32_t)(v0 + k);
            if (v + 1 == sym) lo = quant(acc);
            if (v == sym) hi = quant(acc);
          }
        }
      }
    };
    if (pdf.fast) walk(std::true_type{});
    else walk(std::false_type{});
    __syncwarp();  // (the next column's first group reuses line 0)
    if (kLit && (int)sym >= V) {  // literal symbols follow the vocabulary
      const double pl = pdf.literal();
      for (uint32_t v = (uint32_t)V; v <= sym; v++) {
        acc = __dadd_rn(acc, pl);
        if (v + 1 == sym) lo = quant(acc);
        if (v == sym) hi = quant(acc);
      }
    }
    if (hi < lo) hi = lo;                             // non-decreasing clamp (src/main.rs:818)
    if ((int)sym == n_sym - 1) hi = CZ_AC_CDF_TOTAL;  // cdf[n] = total (src/main.rs:822)
    if (lane == 0) {
      c_lo_out[col] = lo;
      c_hi_out[col] = hi;
    }
  }
}

// K9 from the stats: -log2(max(p_floor(sym), 1e-300)) -- one table lookup per column (src/main.rs:1745-1747 / 1778-1781)
template <int MODE>
__global__ void __launch_bounds__(128) cdf_xe_final_kernel(const float *__restrict__ logits, int V, size_t M, size_t ld,
                                                           const uint32_t *__restrict__ syms, const CdfStats *__restrict__ stats,
                                                           double *__restrict__ xe_out) {
  constexpr bool kLit = MODE == CZ_CDF_RWKV_LITERALS;
  __shared__ uint64_t s_tab[32 * 32];
  exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  const size_t col = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= M) return;
  const int n_sym = kLit ? V + 256 : V;
  const uint32_t sym = syms[col];
  const CdfStats st = stats[col];
  PdfOf<MODE, true> pdf;
  pdf.init(st, V);
  pdf.fast = false;  // a single element: the plain IEEE divisions
  double pr = CZ_P_FLOOR;  // pdf.get(sym).unwrap_or(ac_p_min())
  if ((int)sym < V) {
    const float x = logits[(size_t)sym * ld + col];
    pr = pdf(kLit ? (double)x : (double)cz_expf(__fsub_rn(x, st.mx), tab));
  } else if ((int)sym < n_sym) {
    pr = pdf.literal();
  }
  xe_out[col] = -log2(fmax(pr, 1e-300));
}

// w (30 - log2 w), one term of H below; 0 for w = 0 (the limit: a zero-width symbol contributes nothing).  For w > 2^29 the factor is below 1 and 30 - log2(w) would lose up to 2^-22 of it to cancellation
// (w near 2^30: the coded token of a confident model); -log2(1 - d 2^-30) through log1p keeps it to a few ulp (d = 2^30 - w is exact).
__device__ __forceinline__ double code_len_term(uint32_t w) {
  const double bits = w > (1u << 29) ? __dmul_rn(-log1p(-(double)(CZ_AC_CDF_TOTAL - w) * 0x1p-30), 1.4426950408889634)  // log2(e)
                                     : __dsub_rn(30.0, log2(fmax((double)w, 1.0)));  // (w = 0: 0 x 30, not 0 x inf = NaN)
  return __dmul_rn((double)w, bits);
}

// Expected code length of every column's coding distribution, from the stats the stats pass left:
//   H = 2^-30 sum_{s < n, w_s > 0} w_s (30 - log2 w_s),   w_s = cdf[s + 1] - cdf[s]
// with cdf exactly the coder's (cdf_full_kernel's accumulation, quant, monotone clamp, cdf[n] = 2^30), summed in f64 in ascending s.
// One thread per column (its own sequential walk: no cross-thread reduction, so H is a pure function of the column), direct coalesced
// loads of the vocab-major rows.  The rows hold logits (SmolLM) or the e_v the stats pass left in their slots (RWKV alphabet).  The
// last width is 2^30 - cdf[n - 1], so the last row of the SmolLM alphabets is never read.  A width equal to the previous one reuses its
// term: in the tail of a real distribution the widths repeat, and log2 is the most expensive operation of the walk.
template <int MODE>
__global__ void __launch_bounds__(128) cdf_entropy_kernel(const float *__restrict__ logits, int V, size_t M, size_t ld,
                                                          const CdfStats *__restrict__ stats, double *__restrict__ h_out) {
  constexpr bool kLit = MODE == CZ_CDF_RWKV_LITERALS;
  __shared__ uint64_t s_tab[kLit ? 1 : 32 * 32];
  if (!kLit) exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  const size_t col = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= M) return;
  const CdfStats st = stats[col];
  PdfOf<MODE, MODE == CZ_CDF_SMOLLM_FLOOR> pdf;
  pdf.init(st, V);
  const float mx = st.mx;
  double acc = 0.0, h = 0.0, term = 0.0;
  uint32_t prev = 0, last_w = 0;  // (term = code_len_term(0) = 0)
  auto add = [&](double q) {
    acc = __dadd_rn(acc, q);
    uint32_t cur = quant(acc);
    if (cur < prev) cur = prev;
    const uint32_t w = cur - prev;
    prev = cur;
    if (w != last_w) {
      last_w = w;
      term = code_len_term(w);
    }
    h = __dadd_rn(h, term);
  };
  const int n_rows = kLit ? V : V - 1;
  auto walk = [&](auto fast_tag) {
    constexpr bool kFast = decltype(fast_tag)::value;
    cdf_walk_groups<true>(logits + col, ld, n_rows, [&](int, const float(&x)[CDF_GRP], int cnt) {
      double d[CDF_GRP];
      if (kLit) {
#pragma unroll
        for (int k = 0; k < CDF_GRP; k++) d[k] = kFast ? cz_widen_pos(x[k]) : (double)x[k];  // (values below 2^-126 are floored either way)
      } else {
        float a[CDF_GRP], ef[CDF_GRP];
#pragma unroll
        for (int k = 0; k < CDF_GRP; k++) a[k] = __fsub_rn(mx, x[k]);
        exp_group<CDF_GRP, false>(a, tab, d, ef);
      }
#pragma unroll
      for (int k = 0; k < CDF_GRP; k++)
        if (k < cnt) add(pdf.template get<kFast>(d[k]));
    });
  };
  if (pdf.fast) walk(std::true_type{});
  else walk(std::false_type{});
  if (kLit) {  // literal symbols V .. V + 254 (the last one's width is what is left)
    const double pl = pdf.literal();
    for (int j = 0; j < 255; j++) add(pl);
  }
  const uint32_t w = CZ_AC_CDF_TOTAL - prev;  // cdf[n] = 2^30
  h = __dadd_rn(h, code_len_term(w));
  h_out[col] = __dmul_rn(h, 0x1p-30);
}

// ---- test hooks: the fast paths of cdf_fast.cuh against the originals -----------------------------------------------------------
// every non-negative f32 bit pattern b (a = max - logit >= 0, +inf, NaNs): fast == original wherever exp_group takes the fast path,
// and a checksum of the ORIGINAL expf over the whole domain that the CPU oracle reproduces from glibc-verified code
__global__ void __launch_bounds__(256) expf_exhaustive_kernel(unsigned long long *__restrict__ out /* [0] mismatches [1] checksum [2] first bad */) {
  __shared__ uint64_t s_tab[32 * 32];
  exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  unsigned long long bad = 0, sum = 0, first = ~0ull;
  for (unsigned long long b = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; b < 0x80000000ull; b += (unsigned long long)gridDim.x * blockDim.x) {
    const float a = __uint_as_float((uint32_t)b);
    const float ref = cz_expf(-a, tab);
    uint32_t rb = __float_as_uint(ref);
    if (ref != ref) rb = 0x7fc00000u;
    sum += (unsigned long long)rb * (2ull * b + 1ull);
    if (a <= CZ_EXP_FAST_MAX) {
      const double f = cz_exp_neg_fast(a, tab.t);
      if (__double_as_longlong(f) != __double_as_longlong((double)ref) || __float_as_uint(cz_f32_of_gridded(f)) != __float_as_uint(ref)) {
        bad++;
        if (b < first) first = b;
      }
    }
  }
  atomicAdd(&out[0], bad);
  atomicAdd(&out[1], sum);
  atomicMin(&out[2], first);
}

__device__ __forceinline__ unsigned long long tst_mix(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// cz_div_rcp(a, b, RN(1/b)) == __ddiv_rn(a, b) on random operands of the shapes the CDF passes divide
__global__ void __launch_bounds__(256) div_random_kernel(unsigned long long seed, int iters, unsigned long long *__restrict__ out) {
  unsigned long long st = tst_mix(seed ^ ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 0xD1342543DE82EF95ull);
  unsigned long long bad = 0;
  auto mk = [](unsigned long long mant52, int e) { return __longlong_as_double((long long)(((unsigned long long)(e + 1023) << 52) | (mant52 & 0xFFFFFFFFFFFFFull))); };
  for (int i = 0; i < iters; i++) {
    const unsigned long long r0 = st = tst_mix(st), r1 = st = tst_mix(st), r2 = st = tst_mix(st);
    double a, b;
    switch (i & 7) {
      case 0:
      case 1:  // e / S: e on the f32 grid in [2^-126, 1], S in [1, 2^17)
        a = mk(r0 & 0xFFFFFE0000000ull, -(int)(r2 % 127));
        b = mk(r1, (int)((r2 >> 8) % 17));
        break;
      case 2:  // e near 1 (the tokens that carry the mass), S small
        a = mk(r0 & 0xFFFFFE0000000ull, -(int)(r2 % 4));
        b = mk(r1, (int)((r2 >> 8) % 6));
        break;
      case 3:  // floored q / norm, q / sum2: quotients of doubles near 1
        a = mk(r0, -(int)(r2 % 30));
        b = mk(r1, -(int)((r2 >> 8) % 2));
        break;
      case 4:  // divisor mantissa of all ones / nearly all ones, and just above a power of two
        a = mk(r0, -(int)(r2 % 40));
        b = mk((r2 & 64) ? 0xFFFFFFFFFFFFFull - (r1 & 7) : (r1 & 7), (int)((r2 >> 8) % 17));
        break;
      case 5:  // numerator a multiple of the divisor's leading bits: quotients with long runs of zeros / ones
        b = mk(r1 & 0xFFFFF00000000ull, (int)((r2 >> 8) % 17));
        a = __dmul_rn(b, mk(r0 & 0xFFF0000000000ull, -(int)(r2 % 30)));
        a = __longlong_as_double(__double_as_longlong(a) + (long long)(r2 >> 60) - 8);
        break;
      default:  // anything in the exponent range cz_div_rcp_ok admits
        a = mk(r0, (int)(r2 % 90) - 60);
        b = mk(r1, (int)((r2 >> 8) % 120) - 60);
        break;
    }
    const double y = __drcp_rn(b);
    if (!cz_div_rcp_ok(b)) continue;
    if (__double_as_longlong(cz_div_rcp(a, b, y)) != __double_as_longlong(__ddiv_rn(a, b))) bad++;
  }
  if (bad) atomicAdd(out, bad);
}

// OP_SEARCH for any number of columns (the stepwise decoder runs the same search inside decode_step_kernel, exec.cu):
// cdf_search_warp_n with NC columns per warp (2 here, so that the multi-column form stays covered by the kernel-level parity tests;
// the decoder itself uses 1)
template <int MODE>
__global__ void __launch_bounds__(128) cdf_search_warp_kernel(const float *__restrict__ logits, int V, size_t M, size_t ld,
                                                              const uint32_t *__restrict__ values, uint32_t *__restrict__ sym_out,
                                                              uint32_t *__restrict__ c_lo_out, uint32_t *__restrict__ c_hi_out,
                                                              int *__restrict__ err, const int *__restrict__ colmax) {
  constexpr int NC = 2;
  __shared__ uint64_t s_tab[32 * 32];
  __shared__ __align__(16) double s_xch[4 * NC * 128];  // per warp and column: exchange lines + row ring
  exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  const int warp = threadIdx.x >> 5;
  const size_t col0 = ((size_t)blockIdx.x * 4 + warp) * NC;
  if (col0 >= M) return;
  const float *cp[NC];
  uint32_t value[NC];
  float mx[NC];
  size_t cols[NC];
#pragma unroll
  for (int c = 0; c < NC; c++) {
    const size_t col = col0 + c < M ? col0 + c : col0;  // an odd last column is walked twice
    cols[c] = col;
    cp[c] = logits + col;
    value[c] = values[col];
    if (colmax) {
      mx[c] = colmax_decode(colmax[col]);
    } else {
      float m = __int_as_float(0xff800000);
      for (int v = threadIdx.x & 31; v < V; v += 32) {
        const float x = logits[(size_t)v * ld + col];
        if (x > m) m = x;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      mx[c] = m;
    }
  }
  uint32_t sym[NC], lo[NC], hi[NC];
  int errbits = 0;
  cdf_search_warp_n<MODE, NC>(cp, ld, V, value, mx, tab, sym, lo, hi, errbits, s_xch + warp * (NC * 128));
  if ((threadIdx.x & 31) == 0) {
    if (errbits) atomicOr(err, errbits);
#pragma unroll
    for (int c = 0; c < NC; c++) {
      if (col0 + c >= M) continue;
      sym_out[cols[c]] = sym[c];
      c_lo_out[cols[c]] = lo[c];
      c_hi_out[cols[c]] = hi[c];
    }
  }
}

// full CDF of one column (debug / watchdog parity): single thread, sequential
template <int MODE>
__global__ void cdf_full_kernel(const float *__restrict__ logits, int V, uint32_t *__restrict__ cdf) {
  __shared__ uint64_t s_tab[32 * 32];
  exp_tab64_init(s_tab);
  if (threadIdx.x != 0) return;
  const ExpTab64 tab{s_tab};
  const int n_sym = MODE == CZ_CDF_RWKV_LITERALS ? V + 256 : V;
  float mx = __int_as_float(0xff800000);
  for (int v = 0; v < V; v++)
    if (logits[v] > mx) mx = logits[v];
  double S = 0.0;
  for (int v = 0; v < V; v++) S = __dadd_rn(S, (double)cz_expf(__fsub_rn(logits[v], mx), tab));
  double norm = 1.0, sum2 = 1.0;
  const double scale = 1.0 - 256.0 * CZ_P_FLOOR;
  if (MODE != CZ_CDF_SMOLLM) {
    double acc = 0.0;
    for (int v = 0; v < V; v++)
      acc = __dadd_rn(acc, fmax(__ddiv_rn((double)cz_expf(__fsub_rn(logits[v], mx), tab), S), CZ_P_FLOOR));
    norm = acc;
  }
  if (MODE == CZ_CDF_RWKV_LITERALS) {
    double acc = 0.0;
    for (int v = 0; v < V; v++) {
      double q = fmax(__ddiv_rn((double)cz_expf(__fsub_rn(logits[v], mx), tab), S), CZ_P_FLOOR);
      acc = __dadd_rn(acc, __dmul_rn(__ddiv_rn(q, norm), scale));
    }
    for (int j = 0; j < 256; j++) acc = __dadd_rn(acc, CZ_P_FLOOR);
    sum2 = acc;
  }
  const bool uniform = MODE == CZ_CDF_SMOLLM && S <= 0.0;
  double acc = 0.0;
  uint32_t prev = 0;
  cdf[0] = 0;
  for (int v = 0; v < n_sym; v++) {
    double q;
    if (MODE == CZ_CDF_RWKV_LITERALS) {
      if (v < V) {
        q = fmax(__ddiv_rn((double)cz_expf(__fsub_rn(logits[v], mx), tab), S), CZ_P_FLOOR);
        q = __dmul_rn(__ddiv_rn(q, norm), scale);
      } else {
        q = CZ_P_FLOOR;
      }
      if (sum2 > 0.0) q = __ddiv_rn(q, sum2);
    } else if (MODE == CZ_CDF_SMOLLM_FLOOR) {
      q = __ddiv_rn(fmax(__ddiv_rn((double)cz_expf(__fsub_rn(logits[v], mx), tab), S), CZ_P_FLOOR), norm);
    } else {
      q = uniform ? 1.0 / (double)V : __ddiv_rn((double)cz_expf(__fsub_rn(logits[v], mx), tab), S);
    }
    acc = __dadd_rn(acc, q);
    uint32_t cur = quant(acc);
    if (cur < prev) cur = prev;
    cdf[v + 1] = cur;
    prev = cur;
  }
  cdf[n_sym] = CZ_AC_CDF_TOTAL;
}

__global__ void fill_i32_kernel(int *__restrict__ p, int v, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

}  // namespace czk

namespace cz {

int launch_fill_i32(cz_ctx *ctx, int *p, int v, size_t n, cudaStream_t stream) {
  if (n == 0) return CZ_OK;
  CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::fill_i32_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>(p, v, n)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

// logits [V][ld] f32 as a 2D tensor, box = ST_COLS columns x StCfg<MODE>::ROWS rows, no swizzle (thread t reads word t of a row: conflict-free);
// rows beyond V and columns beyond ld are zero-filled
static int make_logits_map(CUtensorMap *map, const float *logits, size_t V, size_t ld, int box_rows) {
  typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                               CUtensorMapFloatOOBfill);
  static EncodeFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) {
      set_error("cuTensorMapEncodeTiled entry point not available");
      return CZ_ERR_CUDA;
    }
    fn = (EncodeFn)p;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)V};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)czk::ST_COLS, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(logits), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (logits) failed with CUresult " + std::to_string((int)r));
    return CZ_ERR_CUDA;
  }
  return CZ_OK;
}

// Calls f(std::integral_constant<int, MODE>{}) for the coding alphabet `mode`, so that each launch is written once for all of them;
// any other value is CZ_ERR_INVALID.
template <class F>
static int with_cdf_mode(int mode, F &&f) {
  switch (mode) {
    case CZ_CDF_SMOLLM:
      return f(std::integral_constant<int, CZ_CDF_SMOLLM>{});
    case CZ_CDF_RWKV_LITERALS:
      return f(std::integral_constant<int, CZ_CDF_RWKV_LITERALS>{});
    case CZ_CDF_SMOLLM_FLOOR:
      return f(std::integral_constant<int, CZ_CDF_SMOLLM_FLOOR>{});
  }
  set_error("cdf: unknown mode");
  return CZ_ERR_INVALID;
}

// Encode side (OP_BOUNDS / OP_XE): full passes -> per-column stats -> prefix walk / XE lookup
template <int MODE, int OP>
static int launch_cdf_encode(cz_ctx *ctx, const float *logits_dev, size_t V, size_t M, size_t ld, const uint32_t *syms_dev,
                             uint32_t *c_lo_dev, uint32_t *c_hi_dev, double *xe_dev, cudaStream_t stream, const int *colmax_dev) {
  const size_t need = M * sizeof(czk::CdfStats);
  if (need > ctx->cdf_stats_bytes) {
    if (ctx->cdf_stats) {
      CZ_CUDA_TRY(cudaStreamSynchronize(stream));
      cudaFree(ctx->cdf_stats);
      ctx->cdf_stats = nullptr;
      ctx->cdf_stats_bytes = 0;
    }
    const size_t want = need + (need >> 2) + 4096;
    CZ_CUDA_TRY(cudaMalloc(&ctx->cdf_stats, want));
    ctx->cdf_stats_bytes = want;
  }
  czk::CdfStats *stats = (czk::CdfStats *)ctx->cdf_stats;
  float *lg = const_cast<float *>(logits_dev);  // (the RWKV alphabet caches expf in place: the logits batch is scratch)
  // TMA-staged variant: needs tensor-map-compatible strides / alignment and enough columns to fill the machine with 256-column CTAs
  const bool tma_ok = ld % 4 == 0 && ((uintptr_t)logits_dev & 15) == 0 && M >= 256 && V >= 64;
  // e-cache for the prefix walk (see ecache_offsets_kernel): only with the TMA-staged stats kernel, which fills it
  uint32_t *eoff = nullptr;
  double *ecache = nullptr;
  int *eflag = nullptr;
  if (OP == czk::OP_BOUNDS) ctx->cdf_eflag_last = nullptr;
  if (tma_ok && OP == czk::OP_BOUNDS && !ctx->cdf_ecache_failed && getenv("CZ_CDF_NO_ECACHE") == nullptr) {
    const char *env_frac = getenv("CZ_CDF_ECACHE_FRAC");  // (read per call: the tests switch it between calls)
    double frac = env_frac ? atof(env_frac) : 0.25;       // capacity as a fraction of the batch's rows (real text needs 0.1)
    frac = frac < 0.0 ? 0.0 : frac > 1.0 ? 1.0 : frac;
    const size_t grp_per_col = ceil_div(V, (size_t)czk::EC_GRP);
    size_t cap_groups = std::min<size_t>((size_t)((double)M * (double)grp_per_col * frac) + 1, 0xffffffffull);
    const size_t need_e = cap_groups * czk::EC_GRP * sizeof(double), need_o = (M + 2) * sizeof(uint32_t);
    bool ok = true;
    if (need_o > ctx->cdf_eoff_bytes || need_e > ctx->cdf_ecache_bytes) {
      if (ctx->capturing) {
        ok = false;  // no allocation inside a graph capture
      } else {
        CZ_CUDA_TRY(cudaStreamSynchronize(stream));
        if (need_o > ctx->cdf_eoff_bytes) {
          if (ctx->cdf_eoff) cudaFree(ctx->cdf_eoff);
          ctx->cdf_eoff = nullptr;
          ctx->cdf_eoff_bytes = 0;
          const size_t want = need_o + (need_o >> 2) + 4096;
          CZ_CUDA_TRY(cudaMalloc(&ctx->cdf_eoff, want));
          ctx->cdf_eoff_bytes = want;
        }
        if (need_e > ctx->cdf_ecache_bytes) {
          if (ctx->cdf_ecache) cudaFree(ctx->cdf_ecache);
          ctx->cdf_ecache = nullptr;
          ctx->cdf_ecache_bytes = 0;
          if (cudaMalloc(&ctx->cdf_ecache, need_e) != cudaSuccess) {
            cudaGetLastError();  // out of memory: the prefix walk keeps reading the logits, for good
            ctx->cdf_ecache = nullptr;
            ctx->cdf_ecache_failed = true;
            ok = false;
          } else {
            ctx->cdf_ecache_bytes = need_e;
          }
        }
      }
    }
    if (ok) {
      eoff = (uint32_t *)ctx->cdf_eoff;
      eflag = (int *)(eoff + M + 1);
      ecache = (double *)ctx->cdf_ecache;
      const int n_sym = MODE == CZ_CDF_RWKV_LITERALS ? (int)V + 256 : (int)V;
      CZ_LAUNCH(ctx, CZ_K_CDF, (czk::ecache_offsets_kernel<<<1, 1024, 0, stream>>>(syms_dev, M, (int)V, n_sym, eoff, (unsigned long long)cap_groups, eflag)));
      CZ_CHECK_LAUNCH();
      ctx->cdf_eflag_last = eflag;
    }
  }
  if (tma_ok) {
    CUtensorMap tm;
    CZ_TRY(make_logits_map(&tm, logits_dev, V, ld, czk::StCfg<MODE>::ROWS));
    static bool attr = false;
    if (!attr) {
      CZ_CUDA_TRY(cudaFuncSetAttribute(czk::cdf_stats_tma_kernel<MODE, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, czk::StCfg<MODE>::SMEM));
      attr = true;
    }
    const unsigned g = (unsigned)ceil_div(M, (size_t)czk::ST_COLS);
    CZ_LAUNCH(ctx, CZ_K_CDF,
              (czk::cdf_stats_tma_kernel<MODE, OP><<<g, czk::ST_COLS + 32, czk::StCfg<MODE>::SMEM, stream>>>(
                  tm, lg, (int)V, M, ld, colmax_dev, stats, ctx->err_flag_dev, syms_dev, eoff, ecache, eflag)));
  } else {
    const unsigned g = (unsigned)ceil_div(M, 128);
    CZ_LAUNCH(ctx, CZ_K_CDF, (czk::cdf_stats_kernel<MODE, OP><<<g, 128, 0, stream>>>(lg, (int)V, M, ld, colmax_dev, stats, ctx->err_flag_dev)));
  }
  CZ_CHECK_LAUNCH();
  if constexpr (OP == czk::OP_BOUNDS) {
    // persistent warps pulling columns from a counter in the ctx's status block (word 12; the attention kernel's is word 8)
    unsigned int *counter = reinterpret_cast<unsigned int *>(ctx->err_flag_dev + 12);
    CZ_CUDA_TRY(cudaMemsetAsync(counter, 0, sizeof(unsigned int), stream));
    const size_t want_ctas = ceil_div(M, 8);
    const unsigned g = (unsigned)std::min<size_t>(want_ctas, (size_t)ctx->sm_count * 8);
    auto prefix = [&](auto cached) {
      CZ_LAUNCH(ctx, CZ_K_CDF_PREFIX,
                (czk::cdf_bounds_warp_kernel<MODE, decltype(cached)::value><<<g, 256, 0, stream>>>(
                    logits_dev, (int)V, M, ld, syms_dev, stats, c_lo_dev, c_hi_dev, ctx->err_flag_dev, counter, eoff, ecache, eflag)));
    };
    // with an e-cache both variants are issued: the flag the offsets kernel wrote decides on the device which one works
    if (ecache) prefix(std::true_type{});
    prefix(std::false_type{});
  } else {
    const unsigned g = (unsigned)ceil_div(M, 128);
    CZ_LAUNCH(ctx, CZ_K_CDF, (czk::cdf_xe_final_kernel<MODE><<<g, 128, 0, stream>>>(logits_dev, (int)V, M, ld, syms_dev, stats, xe_dev)));
  }
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

// Device-pointer launchers (used by the executor and by the host-buffer C-ABI wrappers in api.cu)
int launch_cdf_cols(cz_ctx *ctx, int op, int mode, const float *logits_dev, size_t V, size_t M, size_t ld,
                    const uint32_t *arg_dev, uint32_t *sym_out_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev,
                    double *xe_dev, cudaStream_t stream, const int *colmax_dev) {
  // OP_XE evaluates the floored pdf for SmolLM whatever the coding alphabet (src/main.rs:1745): mode 2 IS mode 0 there
  if (op == czk::OP_XE && mode == CZ_CDF_SMOLLM_FLOOR) mode = CZ_CDF_SMOLLM;
  return with_cdf_mode(mode, [&](auto mode_c) -> int {
    constexpr int MODE = decltype(mode_c)::value;
    if (M == 0) return CZ_OK;
    if (V == 0 || V > (1u << 24) || ld < M) {
      set_error("cdf: bad shape");
      return CZ_ERR_INVALID;
    }
    if (op == czk::OP_SEARCH) {  // warp per column
      const unsigned g = (unsigned)ceil_div(M, 8);  // 4 warps x 2 columns
      CZ_LAUNCH(ctx, CZ_K_CDF,
                (czk::cdf_search_warp_kernel<MODE><<<g, 128, 0, stream>>>(logits_dev, (int)V, M, ld, arg_dev, sym_out_dev, c_lo_dev, c_hi_dev,
                                                                         ctx->err_flag_dev, colmax_dev)));
      CZ_CHECK_LAUNCH();
      return CZ_OK;
    }
    if constexpr (MODE != CZ_CDF_SMOLLM_FLOOR)  // (mode 2's XE runs as mode 0: no such kernels)
      if (op == czk::OP_XE)
        return launch_cdf_encode<MODE, czk::OP_XE>(ctx, logits_dev, V, M, ld, arg_dev, c_lo_dev, c_hi_dev, xe_dev, stream, colmax_dev);
    return launch_cdf_encode<MODE, czk::OP_BOUNDS>(ctx, logits_dev, V, M, ld, arg_dev, c_lo_dev, c_hi_dev, xe_dev, stream, colmax_dev);
  });
}

// Expected code length of each column (cdf_entropy_kernel).  Reads the per-column stats in ctx->cdf_stats, so it must follow, on the
// same stream, the OP_BOUNDS launch_cdf_cols of the same batch in the same mode (which, in the RWKV alphabet, also left e_v in the
// logits' slots), before anything else overwrites the logits or the stats.
int launch_cdf_entropy(cz_ctx *ctx, int mode, const float *logits_dev, size_t V, size_t M, size_t ld, double *h_dev, cudaStream_t stream) {
  return with_cdf_mode(mode, [&](auto mode_c) -> int {
    if (M == 0) return CZ_OK;
    const unsigned g = (unsigned)ceil_div(M, 128);
    CZ_LAUNCH(ctx, CZ_K_CDF, (czk::cdf_entropy_kernel<decltype(mode_c)::value><<<g, 128, 0, stream>>>(
                                 logits_dev, (int)V, M, ld, (const czk::CdfStats *)ctx->cdf_stats, h_dev)));
    CZ_CHECK_LAUNCH();
    return CZ_OK;
  });
}

int launch_cdf_full(cz_ctx *ctx, int mode, const float *logits_dev, size_t V, uint32_t *cdf_dev, cudaStream_t stream) {
  return with_cdf_mode(mode, [&](auto mode_c) -> int {
    CZ_LAUNCH(ctx, CZ_K_CDF, (czk::cdf_full_kernel<decltype(mode_c)::value><<<1, 32, 0, stream>>>(logits_dev, (int)V, cdf_dev)));
    CZ_CHECK_LAUNCH();
    return CZ_OK;
  });
}

}  // namespace cz

using namespace cz;

extern "C" int cz_test_cdf_ecache_state(cz_ctx *ctx, int *state, uint64_t *groups) {
  if (!ctx || ctx->device < 0) return CZ_ERR_NO_DEVICE;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  CZ_CUDA_TRY(cudaDeviceSynchronize());
  int st = -1;
  uint32_t total = 0;
  if (ctx->cdf_eflag_last) {
    CZ_CUDA_TRY(cudaMemcpy(&st, ctx->cdf_eflag_last, sizeof(int), cudaMemcpyDeviceToHost));
    CZ_CUDA_TRY(cudaMemcpy(&total, (const uint32_t *)ctx->cdf_eflag_last - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  }
  if (state) *state = st;
  if (groups) *groups = total;
  return CZ_OK;
}

extern "C" int cz_test_expf_exhaustive(cz_ctx *ctx, uint64_t *mismatches, uint64_t *checksum, uint64_t *first_bad) {
  if (!ctx || ctx->device < 0) return CZ_ERR_NO_DEVICE;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  unsigned long long *d = nullptr, h[3] = {0, 0, ~0ull};
  CZ_CUDA_TRY(cudaMalloc((void **)&d, 24));
  CZ_CUDA_TRY(cudaMemcpy(d, h, 24, cudaMemcpyHostToDevice));
  czk::expf_exhaustive_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpy(h, d, 24, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) {
    set_error(std::string("expf exhaustive kernel: ") + cudaGetErrorString(e));
    return CZ_ERR_CUDA;
  }
  if (mismatches) *mismatches = h[0];
  if (checksum) *checksum = h[1];
  if (first_bad) *first_bad = h[2];
  return CZ_OK;
}

extern "C" int cz_test_div_random(cz_ctx *ctx, uint64_t seed, uint64_t n_pairs, uint64_t *mismatches) {
  if (!ctx || ctx->device < 0) return CZ_ERR_NO_DEVICE;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  unsigned long long *d = nullptr, h = 0;
  CZ_CUDA_TRY(cudaMalloc((void **)&d, 8));
  CZ_CUDA_TRY(cudaMemset(d, 0, 8));
  const unsigned grid = (unsigned)ctx->sm_count * 8, threads = 256;
  const uint64_t per = n_pairs / ((uint64_t)grid * threads) + 1;
  czk::div_random_kernel<<<grid, threads, 0, ctx->stream>>>(seed, (int)(per > 0x7fffffff ? 0x7fffffff : per), d);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) {
    set_error(std::string("div random kernel: ") + cudaGetErrorString(e));
    return CZ_ERR_CUDA;
  }
  if (mismatches) *mismatches = h;
  return CZ_OK;
}
