// Schedule executor: batched teacher-forced encode, lock-step batched decode, paired XE scan, and the
// batch-of-1 LanguageModelSession shim.  Replaces the per-token loops of src/main.rs:1979-2355 (encode),
// 2528-2653 (decode) and 1725-1751 (gate cross-entropy): logits never leave the GPU, the quantised CDF bounds
// feed the on-device arithmetic-coder lanes directly, and the host only builds row metadata and launches kernels.
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <vector>

#include "cdf_fast.cuh"
#include "coder.cuh"
#include "model.h"
#include "schedule.h"

namespace cz {
int launch_cdf_cols(cz_ctx *ctx, int op, int mode, const float *logits_dev, size_t V, size_t M, size_t ld,
                    const uint32_t *arg_dev, uint32_t *sym_out_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev,
                    double *xe_dev, cudaStream_t stream, const int *colmax_dev = nullptr);
int launch_ac_encode_lanes(cz_ctx *ctx, const uint32_t *c_lo_dev, const uint32_t *c_hi_dev, const uint64_t *lane_off_dev,
                           size_t n_lanes, uint8_t *out_dev, const uint64_t *out_off_dev, uint64_t *out_len_dev,
                           unsigned long long *err_index_dev, cudaStream_t stream, unsigned long long *lane_zw_dev = nullptr);
int require_device(cz_ctx *ctx);
int fetch_device_status(cz_ctx *ctx, unsigned long long *err_index_dev, unsigned long long *err_index_out);
int fetch_device_status_masked(cz_ctx *ctx, unsigned long long *err_index_dev, unsigned long long *err_index_out, int ignore_bits);
// exec_rwkv.cu
int rwkv_encode_bounds(cz_model *m, const uint32_t *ids_dev, const uint32_t *ids_host, size_t n_tokens, const cz_schedule *sched,
                       const uint32_t *extra_dev, const std::vector<size_t> &ev_off, uint32_t *lo_dev, uint32_t *hi_dev, cudaStream_t st);
int rwkv_xe_bits(cz_model *m, const cz_xe_job *jobs, size_t n_jobs, double *bits_out);
int rwkv_chunk_logits(cz_model *m, const uint32_t *prime, size_t prime_len, const uint32_t *targets, size_t n_targets, float *logits_out);
int rwkv_decode(cz_model *m, const uint8_t *payload, const uint64_t *seg_off, size_t n_tokens, const cz_schedule *sched, uint32_t *ids_out);
int rwkv_session_forward(cz_model *m, RwkvState &stt, const uint32_t *tok, size_t n, bool reset, float *logits_dev4, float *logits_out);
}  // namespace cz

namespace czk {

// tok[r] = src[r] >= 0 ? ids[src[r]] : (src[r] == -1 ? bos : extra[-2 - src[r]])
__global__ void gather_tokens_kernel(const long long *__restrict__ src, const uint32_t *__restrict__ ids,
                                     const uint32_t *__restrict__ extra, uint32_t bos, uint32_t *__restrict__ tok, int n) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  long long s = src[r];
  tok[r] = s >= 0 ? ids[s] : (s == -1 ? bos : extra[-2 - s]);
}

__global__ void compact_payload_kernel(const uint8_t *__restrict__ raw, const uint64_t *__restrict__ raw_off,
                                       const uint64_t *__restrict__ dst_off, uint8_t *__restrict__ dst) {
  const uint64_t a = raw_off[blockIdx.x], b = dst_off[blockIdx.x], n = dst_off[blockIdx.x + 1] - b;
  for (uint64_t i = threadIdx.x; i < n; i += blockDim.x) dst[b + i] = raw[a + i];
}

// ---- decode ------------------------------------------------------------------------------------------------
__global__ void ac_decoder_init_kernel(const uint8_t *__restrict__ payload, const uint64_t *__restrict__ seg_off, int n_lanes,
                                       AcDecoderState *__restrict__ st) {
  int lane = blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= n_lanes) return;
  AcDecoder d;
  d.init(payload + seg_off[lane], seg_off[lane + 1] - seg_off[lane]);
  st[lane] = d.s;
}

// One WARP per DS_NC adjacent streams: AC target values -> CDF search over their logits columns (cdf_search_warp_n) -> symbols ->
// AC state updates.  (src/main.rs:2622-2626: to_vec1 + softmax_pdf + quantize_pdf_to_cdf + decode_symbol_counts, fused, on device.)
// 8 warps per CTA take 8 adjacent columns so that the 32-byte sectors of the vocab-major logits are shared through L1.
// DS_NC = 1: two columns per warp (their add chains could fill each other's latency) measured SLOWER on B200 -- 3.18 against 2.87 ms
// per step for the RWKV alphabet at 1,024 streams, 1.70 against 1.44 ms for SmolLM at 1,536 (253 registers, half as many warps).
constexpr int DS_NC = 1, DS_WARPS = 8;
template <int MODE>
__global__ void __launch_bounds__(DS_WARPS * 32) decode_step_kernel(const float *__restrict__ logits, int V, size_t ld, int n_lanes,
                                                                   const uint8_t *__restrict__ payload, const uint64_t *__restrict__ seg_off,
                                                                   const uint64_t *__restrict__ seg_start, uint64_t coded_index,
                                                                   AcDecoderState *__restrict__ st, uint32_t *__restrict__ ids_out,
                                                                   uint32_t *__restrict__ next_tok, int *__restrict__ err,
                                                                   const int *__restrict__ colmax, const unsigned long long *__restrict__ ctr) {
  if (ctr) coded_index = ctr[0];  // device-resident step counter: lets one captured CUDA graph serve every step
  __shared__ uint64_t s_tab[32 * 32];
  __shared__ __align__(16) double s_xch[DS_WARPS * DS_NC * 128];  // per warp and column: exchange lines + row ring (cdf_search_warp_n)
  exp_tab64_init(s_tab);
  const ExpTab64 tab{s_tab + (threadIdx.x & 31)};
  const int warp = threadIdx.x >> 5;
  const int lane0 = (blockIdx.x * DS_WARPS + warp) * DS_NC;  // first stream of this warp (warp-uniform)
  // streams past the batch or past their own end idle (ragged last segments); an idle slot repeats a live stream of the warp
  bool live[DS_NC];
  int stream[DS_NC];
  int any = -1;
#pragma unroll
  for (int c = 0; c < DS_NC; c++) {
    const int l = lane0 + c;
    live[c] = l < n_lanes && coded_index < seg_start[l + 1] - seg_start[l];
    stream[c] = l;
    if (live[c] && any < 0) any = l;
  }
  if (any < 0) return;
  AcDecoder d[DS_NC];
  uint32_t value[DS_NC];
  float mx[DS_NC];
  const float *col[DS_NC];
#pragma unroll
  for (int c = 0; c < DS_NC; c++) {
    if (!live[c]) stream[c] = any;
    const int l = stream[c];
    d[c].resume(st[l], payload + seg_off[l], seg_off[l + 1] - seg_off[l]);
    value[c] = d[c].peek_value();
    col[c] = logits + l;
    if (colmax) {
      mx[c] = colmax_decode(colmax[l]);
    } else {  // engines without the fused column max: parallel max (exact, order-independent)
      float m = __int_as_float(0xff800000);
      for (int v = threadIdx.x & 31; v < V; v += 32) {
        const float x = logits[(size_t)v * ld + l];
        if (x > m) m = x;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      mx[c] = m;
    }
  }
  uint32_t sym[DS_NC], lo[DS_NC], hi[DS_NC];
  int errbits = 0;
  cdf_search_warp_n<MODE, DS_NC>(col, ld, V, value, mx, tab, sym, lo, hi, errbits, s_xch + warp * (DS_NC * 128));
  if ((threadIdx.x & 31) == 0) {
    if (errbits) atomicOr(err, errbits);
#pragma unroll
    for (int c = 0; c < DS_NC; c++) {
      if (!live[c]) continue;
      const int l = stream[c];
      d[c].consume(lo[c], hi[c]);
      st[l] = d[c].s;
      ids_out[seg_start[l] + coded_index] = sym[c];
      next_tok[l] = sym[c];
    }
  }
}

__global__ void fill_int_kernel(int *__restrict__ p, int v, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
// step counters of the lock-step decoder: ctr[0] = coded index, ctr[1] = KV position of the token being fed
__global__ void set_ctr_kernel(unsigned long long *ctr, unsigned long long a, unsigned long long b) {
  ctr[0] = a;
  ctr[1] = b;
}
__global__ void advance_ctr_kernel(unsigned long long *ctr) {
  ctr[0] += 1;
  ctr[1] += 1;
}
__global__ void fill_pos_from_ctr_kernel(int *__restrict__ p, const unsigned long long *__restrict__ ctr, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (int)ctr[1];
}
__global__ void sum_bits_kernel(const double *__restrict__ bits, const uint64_t *__restrict__ job_off, double *__restrict__ out, int n_jobs) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_jobs) return;
  double acc = 0.0;  // sequential f64, like `bits += ...` in src/main.rs:1747
  for (uint64_t t = job_off[j]; t < job_off[j + 1]; t++) acc = __dadd_rn(acc, bits[t]);
  out[j] = acc;
}

}  // namespace czk

namespace cz {

void llama_kernels_set_carveout();
void attn_set_carveout();
static void decode_set_carveout() {
  static bool done = false;
  if (done || !getenv("CZ_CARVEOUT_HINT")) return;  // opt-in experiment: measured no gain on B200 (profiles/decode_r01.md)
  done = true;
  llama_kernels_set_carveout();
  attn_set_carveout();
  const auto mx = cudaSharedmemCarveoutMaxShared;
  cudaFuncSetAttribute(czk::decode_step_kernel<CZ_CDF_SMOLLM>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
  cudaFuncSetAttribute(czk::decode_step_kernel<CZ_CDF_RWKV_LITERALS>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
  cudaFuncSetAttribute(czk::decode_step_kernel<CZ_CDF_SMOLLM_FLOOR>, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
  cudaFuncSetAttribute(czk::fill_pos_from_ctr_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
  cudaFuncSetAttribute(czk::advance_ctr_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, mx);
}
size_t decoder_state_bytes() { return sizeof(czk::AcDecoderState); }
int launch_set_ctr(cz_ctx *ctx, unsigned long long *ctr, unsigned long long a, unsigned long long b, cudaStream_t st) {
  CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::set_ctr_kernel<<<1, 1, 0, st>>>(ctr, a, b)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}
int launch_advance_ctr(cz_ctx *ctx, unsigned long long *ctr, cudaStream_t st) {
  CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::advance_ctr_kernel<<<1, 1, 0, st>>>(ctr)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}
int launch_decoder_init(cz_ctx *ctx, const uint8_t *payload, const uint64_t *seg_off, int n_lanes, void *decoder_state, cudaStream_t st) {
  CZ_LAUNCH(ctx, CZ_K_CODER,
            (czk::ac_decoder_init_kernel<<<(unsigned)ceil_div(n_lanes, 128), 128, 0, st>>>(payload, seg_off, n_lanes,
                                                                                          (czk::AcDecoderState *)decoder_state)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}
int launch_decode_step(cz_ctx *ctx, int mode, const float *logits, int V, size_t ld, int n_lanes, const uint8_t *payload,
                       const uint64_t *seg_off, const uint64_t *seg_start, uint64_t coded_index, void *decoder_state, uint32_t *ids_out,
                       uint32_t *next_tok, const int *colmax, cudaStream_t st, const unsigned long long *ctr) {
  const unsigned grid = (unsigned)ceil_div(n_lanes, czk::DS_NC * czk::DS_WARPS);
  czk::AcDecoderState *ds = (czk::AcDecoderState *)decoder_state;
  if (mode == CZ_CDF_SMOLLM)
    CZ_LAUNCH(ctx, CZ_K_CDF,
              (czk::decode_step_kernel<CZ_CDF_SMOLLM><<<grid, czk::DS_WARPS * 32, 0, st>>>(logits, V, ld, n_lanes, payload, seg_off, seg_start, coded_index, ds,
                                                                            ids_out, next_tok, ctx->err_flag_dev, colmax, ctr)));
  else if (mode == CZ_CDF_RWKV_LITERALS)
    CZ_LAUNCH(ctx, CZ_K_CDF,
              (czk::decode_step_kernel<CZ_CDF_RWKV_LITERALS><<<grid, czk::DS_WARPS * 32, 0, st>>>(logits, V, ld, n_lanes, payload, seg_off, seg_start, coded_index,
                                                                                   ds, ids_out, next_tok, ctx->err_flag_dev, colmax, ctr)));
  else
    CZ_LAUNCH(ctx, CZ_K_CDF,
              (czk::decode_step_kernel<CZ_CDF_SMOLLM_FLOOR><<<grid, czk::DS_WARPS * 32, 0, st>>>(logits, V, ld, n_lanes, payload, seg_off, seg_start, coded_index,
                                                                                  ds, ids_out, next_tok, ctx->err_flag_dev, colmax, ctr)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

// -------------------------------------------------------------------------------------------------------------
// Wave builder: rows of several chunks packed back to back (teacher-forced), each chunk its own sequence.
// -------------------------------------------------------------------------------------------------------------
struct Wave {
  int tile = 64;  // query positions per attention tile (cz_model::attn_tile)
  std::vector<long long> src;
  std::vector<int> pos, kv_base, logit_rows, tile_row0, tile_n;
  size_t n_rows() const { return src.size(); }
  size_t n_tiles() const { return tile_row0.size(); }
  size_t n_logit() const { return logit_rows.size(); }
  void clear() {
    src.clear();
    pos.clear();
    kv_base.clear();
    logit_rows.clear();
    tile_row0.clear();
    tile_n.clear();
  }
  // attention tiles of one sequence occupying rows [base, base + rows): 64 positions each, anchored at position 0
  void add_tiles(int base, int rows) {
    for (int p = 0; p < rows; p += tile) {
      tile_row0.push_back(base + p);
      tile_n.push_back(rows - p < tile ? rows - p : tile);
    }
  }
  // prime_src(k), coded_src(j): token source of prime position k / coded token j
  template <class FP, class FC>
  void add_chunk(uint32_t prime_len, uint32_t n_coded, FP prime_src, FC coded_src) {
    const int base = (int)src.size();
    int p = 0;
    for (uint32_t k = 0; k < prime_len; k++, p++) {
      src.push_back(prime_src(k));
      pos.push_back(p);
      kv_base.push_back(base);
    }
    for (uint32_t j = 0; j + 1 < n_coded; j++, p++) {  // the last coded token is never fed (its logits are unused)
      src.push_back(coded_src(j));
      pos.push_back(p);
      kv_base.push_back(base);
    }
    for (uint32_t j = 0; j < n_coded; j++) logit_rows.push_back(base + (int)prime_len - 1 + (int)j);
    add_tiles(base, p);
  }
};

struct DevBuf {
  void *p = nullptr;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  int alloc(size_t bytes) {
    if (p) cudaFree(p);
    p = nullptr;
    CZ_CUDA_TRY(cudaMalloc(&p, bytes ? bytes : 16));
    return CZ_OK;
  }
  template <class T>
  T *as() { return (T *)p; }
};

// Copies a wave's row metadata through the pinned staging buffer.  The buffer is reused by the next wave, so the
// host waits for the PREVIOUS wave's copies (an event right after them) -- never for the kernels behind them.
static int stage_and_upload(cz_model *m, const Wave &w, long long *src_dev, cudaStream_t st) {
  Workspace &ws = m->ws;
  const size_t R = w.n_rows(), NL = w.n_logit(), NT = w.n_tiles();
  const size_t b_src = R * 8, b_i = R * 4, b_l = NL * 4, b_t = NT * 4;
  if (!ws.stage_ev) CZ_CUDA_TRY(cudaEventCreateWithFlags(&ws.stage_ev, cudaEventDisableTiming));
  else CZ_CUDA_TRY(cudaEventSynchronize(ws.stage_ev));
  CZ_TRY(ensure_stage(m, b_src + 2 * b_i + b_l + 2 * b_t + 64));
  char *h = (char *)ws.h_stage;
  memcpy(h, w.src.data(), b_src);
  memcpy(h + b_src, w.pos.data(), b_i);
  memcpy(h + b_src + b_i, w.kv_base.data(), b_i);
  memcpy(h + b_src + 2 * b_i, w.logit_rows.data(), b_l);
  {
    // Attention work items are pulled from a counter by persistent CTAs.  The tiles keep their natural order (the tiles of a chunk
    // share K / V blocks, which then come out of L2), except that the short ones (at most two key blocks) go to the end of
    // the list: the kernel then ends on 3-6 iteration items instead of a few CTAs still walking 8-block tiles.  The order of
    // the list has no effect on the results (a tile's rows are written by whichever CTA picks it up).
    std::vector<int> order(NT);
    for (size_t t = 0; t < NT; t++) order[t] = (int)t;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      const int la = w.pos[w.tile_row0[a]] + w.tile_n[a] <= 256, lb = w.pos[w.tile_row0[b]] + w.tile_n[b] <= 256;
      return la < lb;
    });
    int *tr = (int *)(h + b_src + 2 * b_i + b_l), *tn = (int *)(h + b_src + 2 * b_i + b_l + b_t);
    for (size_t t = 0; t < NT; t++) {
      tr[t] = w.tile_row0[order[t]];
      tn[t] = w.tile_n[order[t]];
    }
  }
  CZ_CUDA_TRY(cudaMemcpyAsync(src_dev, h, b_src, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.pos, h + b_src, b_i, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.kv_base, h + b_src + b_i, b_i, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, h + b_src + 2 * b_i, b_l, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tile_row0, h + b_src + 2 * b_i + b_l, b_t, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tile_n, h + b_src + 2 * b_i + b_l + b_t, b_t, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaEventRecord(ws.stage_ev, st));
  return CZ_OK;
}

// uploads a wave's metadata, gathers tokens, runs trunk + final norm.  On return ws.xn_logit holds n_logit rows.
static int run_wave_trunk(cz_model *m, const Wave &w, const uint32_t *ids_dev, const uint32_t *extra_dev, uint32_t bos,
                          long long *src_dev_scratch, cudaStream_t st) {
  const size_t R = w.n_rows(), NL = w.n_logit();
  CZ_TRY(ensure_workspace(m, R, NL, w.n_tiles()));
  Workspace &ws = m->ws;
  CZ_TRY(stage_and_upload(m, w, src_dev_scratch, st));
  CZ_LAUNCH(m->ctx, CZ_K_OTHER,
            (czk::gather_tokens_kernel<<<(unsigned)ceil_div(R, 256), 256, 0, st>>>(src_dev_scratch, ids_dev, extra_dev, bos, ws.tok, (int)R)));
  CZ_CHECK_LAUNCH();
  KvView kv;
  kv.k = ws.kpack;
  kv.v = ws.vpack;
  kv.layer_stride = 0;
  kv.n_slots = (int)R;
  kv.tile_row0 = ws.tile_row0;
  kv.tile_n = ws.tile_n;
  kv.n_tiles = (int)w.n_tiles();
  CZ_TRY(forward_trunk(m, (int)R, kv, st));
  CZ_TRY(final_norm_gather(m, (int)NL, st));
  return CZ_OK;
}

// LM head + CDF op over the wave's logit columns, in sub-batches of ws.ld_sub columns.
// syms_dev[j] is the symbol of column j; results go to lo_out/hi_out (OP_BOUNDS) or xe_out (OP_XE), indexed by column.
// digest_first >= 0: the model has a digest sink and column j is coded token digest_first + j (f-4, digest_kernels.cu).
static int run_wave_head(cz_model *m, size_t n_logit, int op, int mode, const uint32_t *syms_dev, uint32_t *lo_out, uint32_t *hi_out,
                         double *xe_out, cudaStream_t st, long long digest_first = -1) {
  CZ_TRY(ensure_logits(m, n_logit));
  Workspace &ws = m->ws;
  cz_ctx *ctx = m->ctx;
  // The CDF pass of a sub-batch (FP64 / integer issue-bound, with a latency-bound tail) runs on the side stream while the main
  // stream goes on with the next sub-batch's LM head or the next wave's trunk (tensor / TMA-bound): different pipes, so part of
  // its time disappears behind them.  Two logits buffers; an event pair per buffer orders LM head -> CDF -> (the LM head that
  // reuses the buffer).  join_cdf() before anything consumes the bounds.
  static const bool no_overlap = getenv("CZ_NO_OVERLAP") != nullptr;  // bisecting aid
  // (per-launch profiling runs everything on one stream: a kernel timed while another one shares the machine says nothing about either)
  const bool overlap = !no_overlap && ctx->stream2 && !ctx->capturing && ctx->prof_mode == 0;
  for (size_t c0 = 0; c0 < n_logit; c0 += ws.ld_sub) {
    const size_t nc = std::min(ws.ld_sub, n_logit - c0);
    const int buf = ws.head_buf;
    ws.head_buf ^= 1;
    int *colmax = ws.colmax + (size_t)buf * ws.ld_sub;
    if (ws.cdf_pending[buf]) {  // the CDF pass that last used this buffer must be done before the LM head overwrites it
      CZ_CUDA_TRY(cudaStreamWaitEvent(st, ws.ev_cdf[buf], 0));
      ws.cdf_pending[buf] = false;
    }
    bool have_max = false;
    CZ_TRY(lm_head(m, (int)c0, (int)nc, ws.logits[buf], ws.ld_sub, st, colmax, &have_max));
    cudaStream_t cst = st;
    if (overlap) {
      cst = ctx->stream2;
      CZ_CUDA_TRY(cudaEventRecord(ws.ev_head[buf], st));
      CZ_CUDA_TRY(cudaStreamWaitEvent(cst, ws.ev_head[buf], 0));
      ctx->prof_stream = cst;
    }
    int rc = CZ_OK;
    if (digest_first >= 0 && m->digest_host)  // (before the CDF pass: the RWKV alphabet's pass overwrites the logits with expf values)
      rc = launch_logits_digest(ctx, ws.logits[buf], (size_t)m->cfg.vocab, nc, ws.ld_sub, m->sb[SB_CV].p, m->sb[SB_DIGEST].as<uint8_t>(),
                                (unsigned long long)digest_first + c0, nullptr, nullptr, nullptr, cst);
    if (rc == CZ_OK)
      rc = launch_cdf_cols(ctx, op, mode, ws.logits[buf], (size_t)m->cfg.vocab, nc, ws.ld_sub, syms_dev + c0, nullptr,
                           lo_out ? lo_out + c0 : nullptr, hi_out ? hi_out + c0 : nullptr, xe_out ? xe_out + c0 : nullptr, cst,
                           have_max ? colmax : nullptr);
    ctx->prof_stream = nullptr;
    CZ_TRY(rc);
    if (overlap) {
      CZ_CUDA_TRY(cudaEventRecord(ws.ev_cdf[buf], cst));
      ws.cdf_pending[buf] = true;
    }
  }
  return CZ_OK;
}

static int check_schedule(const cz_schedule *s, size_t n_tokens) {
  if (!s || s->n_segments == 0 || !s->seg_start || s->seg_start[0] != 0 || s->seg_start[s->n_segments] != n_tokens) {
    set_error("schedule: need n_segments >= 1 and seg_start[0] = 0 .. seg_start[n] = n_tokens");
    return CZ_ERR_INVALID;
  }
  for (uint32_t g = 0; g < s->n_segments; g++)
    if (s->seg_start[g + 1] < s->seg_start[g]) {
      set_error("schedule: seg_start must be non-decreasing");
      return CZ_ERR_INVALID;
    }
  if (s->n_events && s->n_segments != 1) {
    set_error("schedule: hint prime events need n_segments == 1");
    return CZ_ERR_INVALID;
  }
  if (s->reprime_interval == 0 || s->context == 0) {
    set_error("schedule: context and reprime_interval must be > 0");
    return CZ_ERR_INVALID;
  }
  return CZ_OK;
}

// Host-side id validation (ADVICE r1): every id that can reach the embedding table is checked BEFORE anything is launched.
// The limit is the coded alphabet: vocab for SmolLM; vocab + 256 for RWKV-7, whose literal escapes (vocab .. vocab + 255,
// src/main.rs:833-864) never step the model -- they are coded but filtered out of every prime / history (main.rs:1763-1765).
static int check_ids(const uint32_t *ids, size_t n, uint32_t limit, const char *what) {
  for (size_t i = 0; i < n; i++)
    if (ids[i] >= limit) {
      set_error(std::string(what) + ": id " + std::to_string(ids[i]) + " at index " + std::to_string(i) + " is out of range (< " +
                std::to_string(limit) + ")");
      return CZ_ERR_SYMBOL_RANGE;
    }
  return CZ_OK;
}
static uint32_t coded_limit(const cz_model *m) { return (uint32_t)m->cfg.vocab + (m->cfg.arch == CZ_ARCH_RWKV7 ? 256u : 0u); }
static int check_schedule_ids(const cz_model *m, const cz_schedule *s) {
  CZ_TRY(check_ids(&s->bos, 1, (uint32_t)m->cfg.vocab, "schedule bos"));
  for (uint32_t e = 0; e < s->n_events; e++) {
    if (s->events[e].prime_len && !s->events[e].prime) {
      set_error("schedule: prime event without tokens");
      return CZ_ERR_INVALID;
    }
    CZ_TRY(check_ids(s->events[e].prime, s->events[e].prime_len, coded_limit(m), "hint prime token"));
  }
  return CZ_OK;
}

static int arch_mode(const cz_model *m) { return m->cfg.arch == CZ_ARCH_RWKV7 ? CZ_CDF_RWKV_LITERALS : CZ_CDF_SMOLLM; }
// the alphabet cz_encode / cz_decode code with (cz_model_set_pdf_floor only ever sets pdf_floor on a SmolLM model)
static int coded_mode(const cz_model *m) { return m->pdf_floor ? CZ_CDF_SMOLLM_FLOOR : arch_mode(m); }

// Core of cz_encode / cz_encode_dev: ids already on the device.  Leaves the compacted payload in out_dev
// (device) and the per-segment offsets in seg_off_host.
static double host_ms() {
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}

static int encode_core(cz_model *m, const uint32_t *ids_dev, const uint32_t *ids_host, size_t n_tokens, const cz_schedule *sched,
                       uint8_t *out_dev, size_t out_cap, uint64_t *seg_off_host) {
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  static const bool dbg = getenv("CZ_DEBUG_TIMING") != nullptr;
  const double t_begin = host_ms();
  double t_build = 0, t_flush = 0;
  const uint32_t S = sched->n_segments;
  if (m->zw_host && m->zw_cap < S) {
    set_error("zero-width sink too small: " + std::to_string(m->zw_cap) + " < " + std::to_string(S) + " segments");
    return CZ_ERR_INVALID;
  }
  static const size_t env_rows = getenv("CZ_WAVE_ROWS") ? (size_t)atoll(getenv("CZ_WAVE_ROWS")) : 0;  // tuning aid
  const size_t max_rows = sched->max_batch_tokens ? sched->max_batch_tokens : (env_rows ? env_rows : (size_t)262144);
  GrowBuf &d_lo = m->sb[SB_LO], &d_hi = m->sb[SB_HI], &d_src = m->sb[SB_SRC], &d_extra = m->sb[SB_EXTRA], &d_lane = m->sb[SB_LANE],
          &d_raw = m->sb[SB_RAW];
  CZ_TRY(d_lo.reserve(n_tokens * 4, st));
  CZ_TRY(d_hi.reserve(n_tokens * 4, st));
  CZ_TRY(digest_begin(m, n_tokens, 262144, st));
  // explicit prime token lists of the hint events
  std::vector<uint32_t> extra;
  std::vector<size_t> ev_off(sched->n_events + 1, 0);
  for (uint32_t e = 0; e < sched->n_events; e++) {
    ev_off[e] = extra.size();
    extra.insert(extra.end(), sched->events[e].prime, sched->events[e].prime + sched->events[e].prime_len);
  }
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  if (!extra.empty()) CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));

  Wave w;
  w.tile = m->attn_tile;
  size_t wave_first = 0;  // global coded index of the wave's first logit column
  size_t coded_done = 0;
  double t_wave0 = host_ms();
  auto flush = [&]() -> int {
    if (w.n_rows() == 0) return CZ_OK;
    const double t0 = host_ms();
    t_build += t0 - t_wave0;
    CZ_TRY(d_src.reserve(w.n_rows() * 8, st));
    CZ_TRY(run_wave_trunk(m, w, ids_dev, d_extra.as<uint32_t>(), sched->bos, d_src.as<long long>(), st));
    CZ_TRY(run_wave_head(m, w.n_logit(), czk::OP_BOUNDS, coded_mode(m), ids_dev + wave_first, d_lo.as<uint32_t>() + wave_first,
                         d_hi.as<uint32_t>() + wave_first, nullptr, st, m->digest_host ? (long long)wave_first : -1));
    wave_first += w.n_logit();
    w.clear();
    t_wave0 = host_ms();
    t_flush += t_wave0 - t0;
    return CZ_OK;
  };
  std::vector<Chunk> chunks;
  if (m->cfg.arch == CZ_ARCH_RWKV7) {
    CZ_TRY(rwkv_encode_bounds(m, ids_dev, ids_host, n_tokens, sched, d_extra.as<uint32_t>(), ev_off, d_lo.as<uint32_t>(), d_hi.as<uint32_t>(), st));
    coded_done = wave_first = n_tokens;
  }
  for (uint32_t g = 0; g < S && m->cfg.arch != CZ_ARCH_RWKV7; g++) {
    const uint64_t t0 = sched->seg_start[g], n = sched->seg_start[g + 1] - t0;
    build_chunks(n, sched->context, sched->reprime_interval, sched->events, sched->n_events, chunks);
    for (const Chunk &c : chunks) {
      const size_t rows = (size_t)c.prime_len + c.n_coded - 1;
      if (rows > (size_t)m->max_seq()) {
        set_error("schedule produces a sequence longer than the attention kernel supports (" + std::to_string(m->max_seq()) + " positions)");
        return CZ_ERR_UNSUPPORTED;
      }
      if (w.n_rows() + rows > max_rows && w.n_rows() > 0) CZ_TRY(flush());
      // S[k] = k == 0 ? bos : ids[t0 + k - 1];  coded token j of the chunk = ids[t0 + first + j]
      if (c.event >= 0) {
        // prime = tail(S[..=i], hist) ++ explicit tokens, S[0] = BOS, S[k] = ids[t0 + k - 1]
        const long long e0 = (long long)ev_off[c.event];
        const uint32_t hist = c.prime_len - sched->events[c.event].prime_len;
        const uint64_t s0 = c.first + 1 - hist;
        w.add_chunk(c.prime_len, c.n_coded,
                    [&](uint32_t k) {
                      if (k >= hist) return (long long)(-2 - (e0 + (k - hist)));
                      const uint64_t si = s0 + k;
                      return si == 0 ? -1ll : (long long)(t0 + si - 1);
                    },
                    [&](uint32_t j) { return (long long)(t0 + c.first + j); });
      } else {
        w.add_chunk(c.prime_len, c.n_coded,
                    [&](uint32_t k) { uint64_t si = c.prime_start + k; return si == 0 ? -1ll : (long long)(t0 + si - 1); },
                    [&](uint32_t j) { return (long long)(t0 + c.first + j); });
      }
      coded_done += c.n_coded;
    }
  }
  CZ_TRY(flush());
  if (coded_done != n_tokens || wave_first != n_tokens) {
    set_error("internal: schedule did not cover every token");
    return CZ_ERR_INVALID;
  }
  CZ_TRY(join_cdf(m, st));
  // ---- arithmetic-coder lanes: one per segment ----
  std::vector<uint64_t> lane_off(sched->seg_start, sched->seg_start + S + 1), raw_off(S + 1);
  for (uint32_t g = 0; g <= S; g++) raw_off[g] = 4 * lane_off[g] + 8 * (uint64_t)g;
  CZ_TRY(d_lane.reserve((S + 1) * 8 * 5 + 64, st));
  uint64_t *d_lane_off = d_lane.as<uint64_t>(), *d_raw_off = d_lane_off + (S + 1), *d_len = d_raw_off + (S + 1),
           *d_dst_off = d_len + (S + 1);
  unsigned long long *d_eidx = (unsigned long long *)(d_dst_off + (S + 1)), *d_zw = m->zw_host ? d_eidx + 1 : nullptr;
  const unsigned long long none = ~0ull;
  CZ_CUDA_TRY(cudaMemcpyAsync(d_lane_off, lane_off.data(), (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_raw_off, raw_off.data(), (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_eidx, &none, 8, cudaMemcpyHostToDevice, st));
  CZ_TRY(d_raw.reserve(raw_off[S] + 16, st));
  CZ_TRY(launch_ac_encode_lanes(ctx, d_lo.as<uint32_t>(), d_hi.as<uint32_t>(), d_lane_off, S, d_raw.as<uint8_t>(), d_raw_off, d_len,
                                d_eidx, st, d_zw));
  std::vector<uint64_t> len(S);
  CZ_CUDA_TRY(cudaMemcpyAsync(len.data(), d_len, S * 8, cudaMemcpyDeviceToHost, st));
  // with a zero-width sink each lane reports its own first zero-width index there (its payload is left empty) instead of the call failing
  if (d_zw) CZ_CUDA_TRY(cudaMemcpyAsync(m->zw_host, d_zw, S * 8, cudaMemcpyDeviceToHost, st));
  CZ_TRY(fetch_device_status_masked(ctx, d_eidx, nullptr, d_zw ? 4 : 0));
  seg_off_host[0] = 0;
  for (uint32_t g = 0; g < S; g++) seg_off_host[g + 1] = seg_off_host[g] + len[g];
  if (seg_off_host[S] > out_cap) {
    set_error("output buffer too small: need " + std::to_string(seg_off_host[S]) + " bytes");
    return CZ_ERR_NOMEM;
  }
  CZ_CUDA_TRY(cudaMemcpyAsync(d_dst_off, seg_off_host, (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_LAUNCH(ctx, CZ_K_CODER, (czk::compact_payload_kernel<<<S, 128, 0, st>>>(d_raw.as<uint8_t>(), d_raw_off, d_dst_off, out_dev)));
  CZ_CHECK_LAUNCH();
  CZ_TRY(digest_end(m, n_tokens, st));
  const double t_pre_sync = host_ms();
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  if (dbg)
    fprintf(stderr, "[cz timing] encode_core: total %.1f ms | host wave build %.1f | host launch (trunk+head) %.1f | final sync wait %.1f\n",
            host_ms() - t_begin, t_build, t_flush, host_ms() - t_pre_sync);
  return CZ_OK;
}

}  // namespace cz

using namespace cz;

// =============================================================================================================
struct cz_session {
  cz_model *m = nullptr;
  size_t index_pos = 0;
  int max_pos = 1536;
  __nv_bfloat16 *k = nullptr, *v = nullptr;  // [L][max_pos][kvd]
  float *logits_dev = nullptr;               // [V][4]
  long long *src_dev = nullptr;
  uint32_t *hist_dev = nullptr;
  RwkvState rstate;  // RWKV-7: this session's recurrent state (one slot)
};

static int session_forward(cz_session *s, const uint32_t *tok, size_t n, float *logits_out, bool reset = false) {
  cz_model *m = s->m;
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  if (m->cfg.arch == CZ_ARCH_RWKV7) {
    for (size_t i = 0; i < n; i++)
      if (tok[i] >= (uint32_t)m->cfg.vocab) {
        set_error("session: token id out of range");
        return CZ_ERR_SYMBOL_RANGE;
      }
    CZ_TRY(rwkv_session_forward(m, s->rstate, tok, n, reset, s->logits_dev, logits_out));
    s->index_pos = reset ? n : s->index_pos + n;
    return CZ_OK;
  }
  CZ_TRY(check_ids(tok, n, (uint32_t)m->cfg.vocab, "session token"));
  if (s->index_pos + n > (size_t)s->max_pos) {
    set_error("session: KV capacity exceeded");
    return CZ_ERR_INVALID;
  }
  std::vector<int> pos(n), base(n, 0), trow, tn;
  for (size_t i = 0; i < n; i++) pos[i] = (int)(s->index_pos + i);
  if (s->index_pos == 0) {
    for (size_t p = 0; p < n; p += (size_t)m->attn_tile) {
      trow.push_back((int)p);
      tn.push_back((int)std::min<size_t>((size_t)m->attn_tile, n - p));
    }
  } else {  // continuing an existing sequence: one tile per new row (tiles must start at a multiple of 64 or be single rows)
    for (size_t i = 0; i < n; i++) {
      trow.push_back((int)i);
      tn.push_back(1);
    }
  }
  CZ_TRY(ensure_workspace(m, n, 1, trow.size()));
  Workspace &ws = m->ws;
  const int lrow = (int)n - 1;
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tok, tok, n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.pos, pos.data(), n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.kv_base, base.data(), n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, &lrow, 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tile_row0, trow.data(), trow.size() * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tile_n, tn.data(), tn.size() * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));  // pos/base are stack-owned
  KvView kv;
  kv.k = s->k;
  kv.v = s->v;
  kv.layer_stride = (size_t)s->max_pos * m->cfg.n_kv_heads * 64;
  kv.n_slots = s->max_pos;
  kv.tile_row0 = ws.tile_row0;
  kv.tile_n = ws.tile_n;
  kv.n_tiles = (int)trow.size();
  kv.single_rows = s->index_pos != 0;  // continuing a sequence: one tile per new row
  CZ_TRY(forward_trunk(m, (int)n, kv, st));
  CZ_TRY(final_norm_gather(m, 1, st));
  CZ_TRY(lm_head(m, 0, 1, s->logits_dev, 4, st));
  CZ_CUDA_TRY(cudaMemcpy2DAsync(logits_out, 4, s->logits_dev, 16, 4, (size_t)m->cfg.vocab, cudaMemcpyDeviceToHost, st));
  CZ_TRY(fetch_device_status(ctx, nullptr, nullptr));
  s->index_pos += n;
  return CZ_OK;
}

extern "C" {

int cz_session_new(cz_model *m, cz_session **out) {
  if (!m || !out) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(model_finalize(m));
  cz_session *s = new cz_session();
  s->m = m;
  const size_t kvd = (size_t)m->cfg.n_kv_heads * 64, L = m->cfg.n_layers;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (m->cfg.arch == CZ_ARCH_SMOLLM) {
    CZ_CUDA_TRY(cudaMalloc((void **)&s->k, L * s->max_pos * kvd * 2));
    CZ_CUDA_TRY(cudaMalloc((void **)&s->v, L * s->max_pos * kvd * 2));
    CZ_CUDA_TRY(cudaMemset(s->k, 0, L * s->max_pos * kvd * 2));  // unwritten slots must be finite for the masked P V product
    CZ_CUDA_TRY(cudaMemset(s->v, 0, L * s->max_pos * kvd * 2));
  }
  CZ_CUDA_TRY(cudaMalloc((void **)&s->logits_dev, (size_t)m->cfg.vocab * 16));
  *out = s;
  return CZ_OK;
}
void cz_session_free(cz_session *s) {
  if (!s) return;
  cudaSetDevice(s->m->ctx->device);
  cudaDeviceSynchronize();
  if (s->k) cudaFree(s->k);
  if (s->v) cudaFree(s->v);
  if (s->logits_dev) cudaFree(s->logits_dev);
  rwkv_state_free(s->rstate);
  delete s;
}
size_t cz_session_vocab_size(const cz_session *s) { return s ? (size_t)s->m->cfg.vocab : 0; }
size_t cz_session_max_context_length(const cz_session *s) {
  return s && s->m->cfg.arch == CZ_ARCH_SMOLLM ? 512 : (size_t)-1;  // src/models.rs:91, 150
}
size_t cz_session_index_pos(const cz_session *s) { return s ? s->index_pos : 0; }
int cz_session_step_logits(cz_session *s, uint32_t token, float *logits_out) {  // src/models.rs:92-103
  if (!s || !logits_out) return CZ_ERR_INVALID;
  return session_forward(s, &token, 1, logits_out);
}
int cz_session_reprime(cz_session *s, const uint32_t *history, size_t n, float *logits_out) {  // src/models.rs:104-119
  if (!s || !logits_out) return CZ_ERR_INVALID;
  if (n == 0) {
    set_error("reprime called with empty history");
    return CZ_ERR_INVALID;
  }
  s->index_pos = 0;  // fresh KV cache / fresh recurrent state
  return session_forward(s, history, n, logits_out, /*reset=*/true);
}

// -------------------------------------------------------------------------------------------------------------
int cz_encode_dev(cz_model *m, const uint32_t *ids_dev, size_t n_tokens, const cz_schedule *sched, uint8_t *out_dev,
                  size_t out_cap, uint64_t *seg_off_host) {
  if (!m || !seg_off_host) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(check_schedule(sched, n_tokens));
  CZ_TRY(check_schedule_ids(m, sched));  // the coded ids live on the device: the kernels check those (embed / CDF symbol range)
  CZ_TRY(model_finalize(m));
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (n_tokens == 0) {
    // every segment is an empty stream: finish() alone emits 0x40 (1 byte)
  }
  return encode_core(m, ids_dev, nullptr, n_tokens, sched, out_dev, out_cap, seg_off_host);
}

int cz_encode(cz_model *m, const uint32_t *ids, size_t n_tokens, const cz_schedule *sched, cz_bitstreams *out) {
  if (!m || !out || !out->data || !out->seg_off || (n_tokens && !ids)) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(check_schedule(sched, n_tokens));
  CZ_TRY(check_schedule_ids(m, sched));
  CZ_TRY(check_ids(ids, n_tokens, coded_limit(m), "coded token"));
  CZ_TRY(model_finalize(m));
  cz_ctx *ctx = m->ctx;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  GrowBuf &d_ids = m->sb[SB_IDS], &d_out = m->sb[SB_OUT];
  CZ_TRY(d_ids.reserve(n_tokens * 4 + 16, ctx->stream));
  if (n_tokens) CZ_CUDA_TRY(cudaMemcpyAsync(d_ids.p, ids, n_tokens * 4, cudaMemcpyHostToDevice, ctx->stream));
  const size_t cap = 4 * n_tokens + 8 * (size_t)sched->n_segments + 16;
  CZ_TRY(d_out.reserve(cap, ctx->stream));
  CZ_TRY(encode_core(m, d_ids.as<uint32_t>(), ids, n_tokens, sched, d_out.as<uint8_t>(), cap, out->seg_off));
  const uint64_t total = out->seg_off[sched->n_segments];
  if (total > out->cap) {
    set_error("cz_encode: output capacity " + std::to_string(out->cap) + " < payload " + std::to_string(total));
    return CZ_ERR_NOMEM;
  }
  CZ_CUDA_TRY(cudaMemcpyAsync(out->data, d_out.p, total, cudaMemcpyDeviceToHost, ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return CZ_OK;
}

// -------------------------------------------------------------------------------------------------------------
int cz_decode(cz_model *m, const uint8_t *payload, const uint64_t *seg_off, size_t n_tokens, const cz_schedule *sched,
              uint32_t *ids_out) {
  if (!m || !payload || !seg_off || (n_tokens && !ids_out)) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(check_schedule(sched, n_tokens));
  CZ_TRY(check_schedule_ids(m, sched));
  CZ_TRY(model_finalize(m));
  if (n_tokens == 0) return CZ_OK;
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  decode_set_carveout();
  if (m->cfg.arch == CZ_ARCH_RWKV7) return rwkv_decode(m, payload, seg_off, n_tokens, sched, ids_out);
  const cz_model_config &c = m->cfg;
  const uint32_t S = sched->n_segments;
  const size_t kvd = (size_t)c.n_kv_heads * 64, L = c.n_layers;
  uint64_t max_len = 0;
  for (uint32_t g = 0; g < S; g++) max_len = std::max<uint64_t>(max_len, sched->seg_start[g + 1] - sched->seg_start[g]);
  std::vector<Chunk> chunks;  // master timeline = chunk structure of the longest segment
  build_chunks(max_len, sched->context, sched->reprime_interval, sched->events, sched->n_events, chunks);  // events: S == 1
  size_t max_pos = 0;
  for (const Chunk &ch : chunks) max_pos = std::max<size_t>(max_pos, (size_t)ch.prime_len + ch.n_coded);
  max_pos = (max_pos + 63) & ~(size_t)63;
  if (max_pos > (size_t)m->max_seq() + 64) {
    set_error("schedule produces a sequence longer than the attention kernel supports");
    return CZ_ERR_UNSUPPORTED;
  }
  const size_t S_pad = (S + 3) & ~(size_t)3;
  CZ_TRY(ensure_logits(m, S));  // also provides ws.colmax for the fused LM-head column max
  GrowBuf &d_pay = m->sb[SB_PAY], &d_off = m->sb[SB_OFF], &d_start = m->sb[SB_START], &d_state = m->sb[SB_STATE], &d_ids = m->sb[SB_DIDS],
          &d_k = m->sb[SB_K], &d_v = m->sb[SB_V], &d_logits = m->sb[SB_LOGITS], &d_src = m->sb[SB_SRC], &d_kvb = m->sb[SB_KVB];
  const uint64_t pay_total = seg_off[S];
  CZ_TRY(d_pay.reserve(pay_total + 16, st));
  CZ_TRY(d_off.reserve((S + 1) * 8, st));
  CZ_TRY(d_start.reserve((S + 1) * 8, st));
  CZ_TRY(d_state.reserve(S * sizeof(czk::AcDecoderState), st));
  CZ_TRY(d_ids.reserve(n_tokens * 4, st));
  CZ_TRY(d_k.reserve(L * S * max_pos * kvd * 2, st));
  CZ_TRY(d_v.reserve(L * S * max_pos * kvd * 2, st));
  CZ_TRY(d_logits.reserve((size_t)c.vocab * S_pad * 4, st));
  CZ_TRY(digest_begin(m, n_tokens, S, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_pay.p, payload, pay_total, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_off.p, seg_off, (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_start.p, sched->seg_start, (S + 1) * 8, cudaMemcpyHostToDevice, st));
  // explicit prime token lists of the gated hint events (src/main.rs:2586-2614)
  std::vector<uint32_t> extra;
  std::vector<size_t> ev_off(sched->n_events + 1, 0);
  for (uint32_t e = 0; e < sched->n_events; e++) {
    ev_off[e] = extra.size();
    extra.insert(extra.end(), sched->events[e].prime, sched->events[e].prime + sched->events[e].prime_len);
  }
  GrowBuf &d_extra = m->sb[SB_EXTRA];
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  if (!extra.empty()) CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));
  CZ_LAUNCH(ctx, CZ_K_CODER,
            (czk::ac_decoder_init_kernel<<<(unsigned)ceil_div(S, 128), 128, 0, st>>>(d_pay.as<uint8_t>(), d_off.as<uint64_t>(), (int)S,
                                                                                    d_state.as<czk::AcDecoderState>())));
  CZ_CHECK_LAUNCH();
  KvView kv;
  kv.k = d_k.as<__nv_bfloat16>();
  kv.v = d_v.as<__nv_bfloat16>();
  kv.layer_stride = (size_t)S * max_pos * kvd;
  if (m->attn_tc) {  // unwritten slots inside a 128-key block are masked (P = 0), but 0 * NaN = NaN: they must hold finite values
    CZ_CUDA_TRY(cudaMemsetAsync(d_v.p, 0, L * S * max_pos * kvd * 2, st));
    CZ_CUDA_TRY(cudaMemsetAsync(d_k.p, 0, L * S * max_pos * kvd * 2, st));
  }
  kv.n_slots = (int)(S * max_pos);
  Wave w;
  w.tile = m->attn_tile;
  // per-stream constant metadata for the single-token steps
  std::vector<int> kvb(S), lrows(S);
  for (uint32_t g = 0; g < S; g++) {
    kvb[g] = (int)(g * max_pos);
    lrows[g] = (int)g;
  }
  CZ_TRY(d_kvb.reserve(S * 12 + 64, st));
  int *d_kvb_i = d_kvb.as<int>(), *d_lrows_i = d_kvb_i + S, *d_ones_i = d_lrows_i + S;  // step tiles: row0 = g, n = 1
  unsigned long long *d_ctr = (unsigned long long *)(d_kvb.as<char>() + (((size_t)S * 12 + 15) & ~(size_t)15));
  const bool use_graph = getenv("CZ_DECODE_NO_GRAPH") == nullptr;
  std::vector<int> ones(S, 1);
  CZ_CUDA_TRY(cudaMemcpyAsync(d_kvb_i, kvb.data(), S * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_lrows_i, lrows.data(), S * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_ones_i, ones.data(), S * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));

  bool have_max = false;
  for (const Chunk &ch : chunks) {
    // ---- prime every stream that is still live at this chunk (fresh cache: positions 0 .. prime_len-1) ----
    std::vector<uint32_t> live;
    for (uint32_t g = 0; g < S; g++)
      if (sched->seg_start[g + 1] - sched->seg_start[g] > ch.first) live.push_back(g);
    if (live.empty()) break;
    // column g of the logits must be stream g: live streams have to be the prefix [0, n_live), i.e. segment
    // lengths non-increasing (the host splitter puts the longer segments first)
    for (size_t i = 0; i < live.size(); i++)
      if (live[i] != i) {
        set_error("cz_decode: segment lengths must be non-increasing (longest first) for the lock-step decoder");
        return CZ_ERR_UNSUPPORTED;
      }
    w.clear();
    for (uint32_t g : live) {
      const uint64_t t0 = sched->seg_start[g];
      const int base = (int)(g * max_pos);
      const int r0 = (int)w.src.size();
      for (uint32_t k = 0; k < ch.prime_len; k++) {
        const uint64_t si = ch.prime_start + k;
        if (ch.event >= 0) {  // tail of what this stream has decoded so far, then the explicit hint tokens
          const uint32_t hist = ch.prime_len - sched->events[ch.event].prime_len;
          const uint64_t sh = ch.first + 1 - hist + k;
          if (k >= hist) w.src.push_back(-2 - (long long)(ev_off[ch.event] + (k - hist)));
          else w.src.push_back(sh == 0 ? -1ll : (long long)(t0 + sh - 1));
        } else {
          w.src.push_back(si == 0 ? -1ll : (long long)(t0 + si - 1));
        }
        w.pos.push_back((int)k);
        w.kv_base.push_back(base);
      }
      w.logit_rows.push_back((int)w.src.size() - 1);
      w.add_tiles(r0, (int)ch.prime_len);
    }
    {
      const size_t R = w.n_rows(), NL = w.n_logit();
      CZ_TRY(d_src.reserve(R * 8, st));
      CZ_TRY(ensure_workspace(m, std::max<size_t>(R, S), std::max<size_t>(NL, S), std::max<size_t>(w.n_tiles(), S)));
      Workspace &ws = m->ws;
      CZ_TRY(stage_and_upload(m, w, d_src.as<long long>(), st));
      CZ_LAUNCH(ctx, CZ_K_OTHER,
                (czk::gather_tokens_kernel<<<(unsigned)ceil_div(R, 256), 256, 0, st>>>(d_src.as<long long>(), d_ids.as<uint32_t>(),
                                                                                      d_extra.as<uint32_t>(), sched->bos, ws.tok, (int)R)));
      CZ_CHECK_LAUNCH();
      kv.tile_row0 = ws.tile_row0;
      kv.tile_n = ws.tile_n;
      kv.n_tiles = (int)w.n_tiles();
      kv.single_rows = false;
      CZ_TRY(forward_trunk(m, (int)R, kv, st));
      CZ_TRY(final_norm_gather(m, (int)NL, st));
      CZ_TRY(lm_head(m, 0, (int)NL, d_logits.as<float>(), S_pad, st, ws.colmax, &have_max));
    }
    const int n_live = (int)live.size();
    Workspace &ws = m->ws;
    // per-chunk constants of the single-token steps: row g = stream g, one attention tile per row
    CZ_CUDA_TRY(cudaMemcpyAsync(ws.kv_base, d_kvb_i, (size_t)n_live * 4, cudaMemcpyDeviceToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, d_lrows_i, (size_t)n_live * 4, cudaMemcpyDeviceToDevice, st));
    kv.tile_row0 = d_lrows_i;
    kv.tile_n = d_ones_i;
    kv.n_tiles = n_live;
    kv.single_rows = true;
    CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::set_ctr_kernel<<<1, 1, 0, st>>>(d_ctr, ch.first, ch.prime_len)));
    CZ_CHECK_LAUNCH();
    // one step: decode the symbol of every live stream from its logits column, then feed it back (a single-token
    // forward at position ctr[1]) to get the next logits.  All step-varying scalars live in d_ctr, so the same
    // sequence of ~250 launches is captured ONCE per chunk into a CUDA graph and replayed (the eager loop is
    // launch-bound: ~15 us of host work per launch against ~2 us of device work).
    auto decode_syms = [&]() -> int {
      if (m->digest_host)  // f-4: digest of the logits each live stream is about to decode from, at index seg_start[g] + ctr[0]
        CZ_TRY(launch_logits_digest(ctx, d_logits.as<float>(), (size_t)c.vocab, (size_t)n_live, S_pad, m->sb[SB_CV].p,
                                    m->sb[SB_DIGEST].as<uint8_t>(), 0, nullptr, d_start.as<uint64_t>(), d_ctr, st));
      return launch_decode_step(ctx, coded_mode(m), d_logits.as<float>(), c.vocab, S_pad, n_live, d_pay.as<uint8_t>(), d_off.as<uint64_t>(),
                                d_start.as<uint64_t>(), 0, d_state.p, d_ids.as<uint32_t>(), ws.tok, have_max ? ws.colmax : nullptr, st, d_ctr);
    };
    auto step = [&]() -> int {
      CZ_TRY(decode_syms());
      CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::fill_pos_from_ctr_kernel<<<(unsigned)ceil_div(n_live, 256), 256, 0, st>>>(ws.pos, d_ctr, n_live)));
      CZ_CHECK_LAUNCH();
      CZ_TRY(forward_trunk(m, n_live, kv, st));
      CZ_TRY(final_norm_gather(m, n_live, st));
      CZ_TRY(lm_head(m, 0, n_live, d_logits.as<float>(), S_pad, st, ws.colmax, &have_max));
      CZ_LAUNCH(ctx, CZ_K_OTHER, (czk::advance_ctr_kernel<<<1, 1, 0, st>>>(d_ctr)));
      CZ_CHECK_LAUNCH();
      return CZ_OK;
    };
    const uint32_t n_steps = ch.n_coded - 1;  // the step after the chunk's last symbol is never used (next chunk re-primes)
    cudaGraphExec_t gexec = nullptr;
    uint64_t nodes = 0;
    int rc = CZ_OK;
    for (uint32_t j = 0; j < n_steps && rc == CZ_OK; j++) {
      if (j == 0 || !use_graph || n_steps < 4) {
        rc = step();  // first step eager: warms function attributes / lazy allocations outside any capture
      } else if (!gexec) {
        cudaGraph_t graph = nullptr;
        const uint64_t l0 = ctx->launches;
        ctx->capturing = true;
        cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed);
        if (e == cudaSuccess) {
          rc = step();
          e = cudaStreamEndCapture(st, &graph);
        }
        ctx->capturing = false;
        nodes = ctx->launches - l0;
        if (rc == CZ_OK && e == cudaSuccess) e = cudaGraphInstantiate(&gexec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (rc == CZ_OK && e != cudaSuccess) {
          set_error(std::string("decode step graph capture failed: ") + cudaGetErrorString(e));
          rc = CZ_ERR_CUDA;
        }
        if (rc == CZ_OK && cudaGraphLaunch(gexec, st) != cudaSuccess) rc = CZ_ERR_CUDA;
      } else {
        if (cudaGraphLaunch(gexec, st) != cudaSuccess) {
          set_error("cudaGraphLaunch failed");
          rc = CZ_ERR_CUDA;
        }
        ctx->launches += nodes;
      }
    }
    if (gexec) cudaGraphExecDestroy(gexec);
    CZ_TRY(rc);
    CZ_TRY(decode_syms());  // the chunk's last symbol
    CZ_TRY(fetch_device_status(ctx, nullptr, nullptr));
  }
  CZ_CUDA_TRY(cudaMemcpyAsync(ids_out, d_ids.p, n_tokens * 4, cudaMemcpyDeviceToHost, st));
  CZ_TRY(digest_end(m, n_tokens, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  return CZ_OK;
}

// -------------------------------------------------------------------------------------------------------------
int cz_xe_bits(cz_model *m, const cz_xe_job *jobs, size_t n_jobs, double *bits_out) {
  if (!m || (n_jobs && (!jobs || !bits_out))) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(model_finalize(m));
  if (n_jobs == 0) return CZ_OK;
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  for (size_t j = 0; j < n_jobs; j++) {
    if ((jobs[j].prime_len && !jobs[j].prime) || (jobs[j].n_targets && !jobs[j].targets)) return CZ_ERR_INVALID;
    CZ_TRY(check_ids(jobs[j].prime, jobs[j].prime_len, coded_limit(m), "xe prime token"));
    CZ_TRY(check_ids(jobs[j].targets, jobs[j].n_targets, coded_limit(m), "xe target"));
  }
  if (m->cfg.arch == CZ_ARCH_RWKV7) return rwkv_xe_bits(m, jobs, n_jobs, bits_out);
  // all tokens go to the `extra` buffer: [prime_0 | targets_0 | prime_1 | targets_1 | ...]; a parallel buffer holds
  // the targets contiguously in job order so that column j's symbol is tgt[j]
  std::vector<uint32_t> extra, tgt;
  std::vector<uint64_t> job_off(n_jobs + 1, 0);
  std::vector<size_t> p_off(n_jobs), t_off(n_jobs);
  for (size_t j = 0; j < n_jobs; j++) {
    if (jobs[j].n_targets && jobs[j].prime_len == 0) {
      set_error("xe job with targets needs a non-empty prime (the reference bails on an empty reprime)");
      return CZ_ERR_INVALID;
    }
    p_off[j] = extra.size();
    extra.insert(extra.end(), jobs[j].prime, jobs[j].prime + jobs[j].prime_len);
    t_off[j] = extra.size();
    extra.insert(extra.end(), jobs[j].targets, jobs[j].targets + jobs[j].n_targets);
    tgt.insert(tgt.end(), jobs[j].targets, jobs[j].targets + jobs[j].n_targets);
    job_off[j + 1] = job_off[j] + jobs[j].n_targets;
  }
  const size_t n_cols = tgt.size();
  GrowBuf &d_extra = m->sb[SB_EXTRA], &d_tgt = m->sb[SB_TGT], &d_bits = m->sb[SB_BITS], &d_src = m->sb[SB_SRC], &d_joff = m->sb[SB_JOFF],
          &d_out = m->sb[SB_XOUT];
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  CZ_TRY(d_tgt.reserve(n_cols * 4 + 16, st));
  CZ_TRY(d_bits.reserve(n_cols * 8 + 16, st));
  CZ_TRY(d_joff.reserve((n_jobs + 1) * 8, st));
  CZ_TRY(d_out.reserve(n_jobs * 8, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));
  if (n_cols) CZ_CUDA_TRY(cudaMemcpyAsync(d_tgt.p, tgt.data(), n_cols * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_joff.p, job_off.data(), (n_jobs + 1) * 8, cudaMemcpyHostToDevice, st));
  const size_t max_rows = 262144;
  size_t col_first = 0;
  Wave w;
  w.tile = m->attn_tile;
  auto flush = [&]() -> int {
    if (w.n_rows() == 0) return CZ_OK;
    CZ_TRY(d_src.reserve(w.n_rows() * 8, st));
    CZ_TRY(run_wave_trunk(m, w, nullptr, d_extra.as<uint32_t>(), 0, d_src.as<long long>(), st));
    CZ_TRY(run_wave_head(m, w.n_logit(), czk::OP_XE, arch_mode(m), d_tgt.as<uint32_t>() + col_first, nullptr, nullptr,
                         d_bits.as<double>() + col_first, st));
    col_first += w.n_logit();
    w.clear();
    return CZ_OK;
  };
  for (size_t j = 0; j < n_jobs; j++) {
    if (jobs[j].n_targets == 0) continue;
    const size_t rows = (size_t)jobs[j].prime_len + jobs[j].n_targets - 1;
    if (rows > (size_t)m->max_seq()) {
      set_error("xe job longer than the attention kernel supports");
      return CZ_ERR_UNSUPPORTED;
    }
    if (w.n_rows() + rows > max_rows && w.n_rows() > 0) CZ_TRY(flush());
    const long long p0 = (long long)p_off[j], t0 = (long long)t_off[j];
    w.add_chunk(jobs[j].prime_len, jobs[j].n_targets, [&](uint32_t k) { return -2 - (p0 + k); }, [&](uint32_t q) { return -2 - (t0 + q); });
  }
  CZ_TRY(flush());
  CZ_TRY(join_cdf(m, st));
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::sum_bits_kernel<<<(unsigned)ceil_div(n_jobs, 128), 128, 0, st>>>(d_bits.as<double>(), d_joff.as<uint64_t>(),
                                                                                  d_out.as<double>(), (int)n_jobs)));
  CZ_CHECK_LAUNCH();
  CZ_CUDA_TRY(cudaMemcpyAsync(bits_out, d_out.p, n_jobs * 8, cudaMemcpyDeviceToHost, st));
  return fetch_device_status(ctx, nullptr, nullptr);
}

int cz_chunk_logits(cz_model *m, const uint32_t *prime, size_t prime_len, const uint32_t *targets, size_t n_targets,
                    float *logits_out) {
  if (!m || !prime || !prime_len || !n_targets || !logits_out) return CZ_ERR_INVALID;
  CZ_TRY(require_device(m->ctx));
  CZ_TRY(model_finalize(m));
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  if (!targets) return CZ_ERR_INVALID;
  CZ_TRY(check_ids(prime, prime_len, coded_limit(m), "chunk prime token"));
  CZ_TRY(check_ids(targets, n_targets, coded_limit(m), "chunk target"));
  if (m->cfg.arch == CZ_ARCH_RWKV7) return rwkv_chunk_logits(m, prime, prime_len, targets, n_targets, logits_out);
  std::vector<uint32_t> extra(prime, prime + prime_len);
  if (n_targets > 1) extra.insert(extra.end(), targets, targets + n_targets - 1);
  GrowBuf &d_extra = m->sb[SB_EXTRA], &d_src = m->sb[SB_SRC];
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));
  Wave w;
  w.tile = m->attn_tile;
  w.add_chunk((uint32_t)prime_len, (uint32_t)n_targets, [&](uint32_t k) { return -2 - (long long)k; },
              [&](uint32_t q) { return -2 - (long long)(prime_len + q); });
  CZ_TRY(d_src.reserve(w.n_rows() * 8, st));
  CZ_TRY(run_wave_trunk(m, w, nullptr, d_extra.as<uint32_t>(), 0, d_src.as<long long>(), st));
  CZ_TRY(ensure_logits(m, 256));
  Workspace &ws = m->ws;
  const size_t V = m->cfg.vocab;
  const size_t ld_c = std::min<size_t>(ws.ld_sub, 256);  // small sub-batches: this is a test / debugging entry point
  std::vector<float> tmp(V * ld_c);
  for (size_t c0 = 0; c0 < n_targets; c0 += ld_c) {
    const size_t nc = std::min(ld_c, n_targets - c0);
    CZ_TRY(lm_head(m, (int)c0, (int)nc, ws.logits[0], ld_c, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(tmp.data(), ws.logits[0], V * ld_c * 4, cudaMemcpyDeviceToHost, st));
    CZ_CUDA_TRY(cudaStreamSynchronize(st));
    for (size_t j = 0; j < nc; j++)
      for (size_t v = 0; v < V; v++) logits_out[(c0 + j) * V + v] = tmp[v * ld_c + j];
  }
  return fetch_device_status(ctx, nullptr, nullptr);
}

}  // extern "C"
