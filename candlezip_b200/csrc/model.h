// Internal model representation (SmolLM / LLaMA architecture; RWKV-7 shares the tensor store).
#pragma once
#include <string>
#include <unordered_map>
#include <vector>

#include "cz_common.cuh"

struct TensorSlot {
  std::string name;
  size_t n = 0;
  std::vector<uint16_t> host;        // bf16 bits; kept only on host-only ctxs (device ctxs read back on demand)
  __nv_bfloat16 *dev = nullptr;
  bool set = false;
};

struct Workspace {
  size_t cap_rows = 0, cap_logit = 0;
  float *x = nullptr;                 // [rows][D]   residual stream, fp32
  __nv_bfloat16 *xn = nullptr;        // [rows][D]   normed activations (GEMM A operand); fused-norm path: bf16(x * w_norm), unscaled
  float *ssq = nullptr;               // [rows][12]  fused-norm path: per-row partial sums of x^2 (see EPI_ADD_NORM)
  float *qkv = nullptr;               // [rows][(nh+2nkv)*64]
  __nv_bfloat16 *q = nullptr;         // [rows][D]
  __nv_bfloat16 *attn = nullptr;      // [rows][D]
  __nv_bfloat16 *act = nullptr;       // [rows][F]
  __nv_bfloat16 *kpack = nullptr;     // packed-mode (teacher-forced) K rows of the current layer [rows][kvd]
  __nv_bfloat16 *vpack = nullptr;
  uint32_t *tok = nullptr;            // row metadata
  int *pos = nullptr;
  int *kv_base = nullptr;
  int *tile_row0 = nullptr;           // attention tiles: first row / number of valid positions (<= 64), [cap_rows/64 + ...]
  int *tile_n = nullptr;
  size_t cap_tiles = 0;
  int *logit_rows = nullptr;          // [cap_logit]
  uint32_t *syms = nullptr;           // [cap_logit] symbol coded from each logit row
  uint64_t *out_index = nullptr;      // [cap_logit] global coded index the result belongs to
  __nv_bfloat16 *xn_logit = nullptr;  // [cap_logit][D]
  uint32_t *lo_tmp = nullptr, *hi_tmp = nullptr;  // [sub] per-sub-batch CDF outputs before the scatter
  double *xe_tmp = nullptr;
  int *colmax = nullptr;              // [ld_sub] per-column max of the current logits sub-batch (buffer 0; buffer 1 follows it)
  float *logits[2] = {nullptr, nullptr};  // [V][ld_sub] vocab-major, double-buffered: the CDF pass of one sub-batch runs on the
                                          // side stream while the main stream already computes the next wave / sub-batch
  size_t ld_sub = 0;
  int head_buf = 0;                   // logits buffer the next LM-head launch writes
  cudaEvent_t ev_head[2] = {nullptr, nullptr}, ev_cdf[2] = {nullptr, nullptr};
  bool cdf_pending[2] = {false, false};  // a CDF pass on the side stream still owns that buffer
  // pinned host staging for row metadata
  void *h_stage = nullptr;
  size_t h_stage_bytes = 0;
  cudaEvent_t stage_ev = nullptr;
};

// grow-only device buffer owned by the model: API calls are synchronous, so scratch is reused call to call instead of
// paying cudaMalloc/cudaFree (tens of ms, far worse while anything polls the driver) on every encode/decode
struct GrowBuf {
  void *p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes, cudaStream_t st);
  template <class T>
  T *as() { return (T *)p; }
};
enum { SB_LO = 0, SB_HI, SB_SRC, SB_EXTRA, SB_LANE, SB_RAW, SB_IDS, SB_OUT, SB_PAY, SB_OFF, SB_START, SB_STATE, SB_DIDS, SB_K, SB_V,
       SB_LOGITS, SB_KVB, SB_TGT, SB_BITS, SB_JOFF, SB_XOUT, SB_RW_OIDX, SB_RW_SYMS, SB_RW_LO, SB_RW_HI, SB_RW_XE, SB_RW_FRESH,
       SB_DIGEST, SB_CV, SB_ENT, SB_MATCH, SB_MTEMP, SB_MDEC, SB_MOUT,
       SB_COUNT };

// ---- RWKV-7 (rwkv7.cu) ----
enum { RV_PRE_W = 0, RV_PRE_B, RV_LN1_W, RV_LN1_B, RV_LN2_W, RV_LN2_B, RV_XR, RV_XW, RV_XK, RV_XV, RV_XA, RV_XG, RV_KK, RV_KA, RV_RK,
       RV_W0, RV_A0, RV_V0, RV_GNW, RV_GNB, RV_FXK, RV_COUNT };
struct RwkvLayerW {
  __nv_bfloat16 *wr, *wk, *wv, *wo, *w1, *w2, *a1, *a2, *v1, *v2, *g1, *g2, *fk, *fv;
};
struct RwkvWeights {
  std::vector<RwkvLayerW> layers;
  float *vecs = nullptr;            // [L][RV_COUNT][C] + ln_out weight, bias
  __nv_bfloat16 *v_pad = nullptr;   // v-LoRA matrices zero-padded to rank 64
};
struct RwkvWs {
  size_t cap_rows = 0, cap_streams = 0;
  __nv_bfloat16 *mix[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // xr xw xk xv xa xg  [rows][C]
  float *f[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // r k v w-lora a-lora v-lora g  [rows][C]
  float *v_first = nullptr;        // [rows][C]
  __nv_bfloat16 *lo = nullptr;     // [rows][128] LoRA bottleneck activations
  __nv_bfloat16 *att = nullptr;    // [rows][C]
  __nv_bfloat16 *act = nullptr;    // [rows][F]
  int *prev_row = nullptr, *slot = nullptr, *flags = nullptr;         // per row
  int *row_begin = nullptr, *row_end = nullptr, *stream_slot = nullptr;  // per stream of the slab
};
// recurrent state of `cap` stream slots: WKV state + the two token-shift rows per layer (rwkv7.rs:35-61)
struct RwkvState {
  size_t cap = 0, n = 0;
  float *S = nullptr;                       // [L][cap][H][4096], (j/4, i, j%4) order inside a head
  float *xa[2] = {nullptr, nullptr};        // [L][cap][C] attention token shift, ping-pong across slabs
  float *xf[2] = {nullptr, nullptr};        // [L][cap][C] feed-forward token shift
  int cur = 0;
};

struct cz_model {
  GrowBuf sb[SB_COUNT];
  RwkvWeights rw;
  RwkvWs rws;
  RwkvState rstate;
  __nv_bfloat16 *head_w = nullptr;  // LM head [V][D] (SmolLM: tied to the embedding)
  cz_ctx *ctx = nullptr;
  cz_model_config cfg;
  std::vector<TensorSlot> tensors;
  std::unordered_map<std::string, int> index;
  bool finalized = false;
  // packed device weights (SmolLM)
  __nv_bfloat16 *w_qkv = nullptr;  // [L][(nh+2nkv)*64][D]
  __nv_bfloat16 *w_o = nullptr;    // [L][D][D]
  __nv_bfloat16 *w_gu = nullptr;   // [L][2F][D], gate/up interleaved in groups of gu_bn/2 rows
  __nv_bfloat16 *w_d = nullptr;    // [L][D][F]
  __nv_bfloat16 *embed = nullptr;  // alias of the embed_tokens slot
  float *norms = nullptr;          // [L][2][D] + [D]
  float *cos_tab = nullptr, *sin_tab = nullptr;  // [rope_max_pos][32]
  int rope_max_pos = 8192;  // SmolLM2 max_position_embeddings
  // longest sequence (prime + coded tokens of one chunk) the attention kernel in use can take
  int max_seq() const { return attn_tc ? rope_max_pos - 1 : 2000; }
  int gu_bn = 192;
  bool attn_tc = false;  // tcgen05 attention kernel (attn_tc.cu); else the mma.sync kernel (attn_mma.cu)
  int attn_tile = 64;    // query positions per attention tile (128 with attn_tc)
  Workspace ws;
  // f-4 watchdog digests (digest_kernels.cu): when set, every coded token's logits vector is hashed on the device during
  // cz_encode / cz_encode_dev / cz_decode and the 16-byte digests are copied here (index = global coded index)
  uint8_t *digest_host = nullptr;
  size_t digest_cap = 0;
  // cz_model_set_pdf_floor: SmolLM streams are coded with CZ_CDF_SMOLLM_FLOOR (exec.cu, coded_mode)
  bool pdf_floor = false;
  // cz_model_set_zero_width_out: per-segment first zero-width index of cz_encode / cz_encode_dev (exec.cu, encode_core)
  uint64_t *zw_host = nullptr;
  size_t zw_cap = 0;
  // cz_model_set_code_length_out: per-token interval and coding-distribution entropy of cz_encode / cz_encode_dev (exec.cu, encode_core)
  uint32_t *cl_lo_host = nullptr, *cl_hi_host = nullptr;
  double *cl_ent_host = nullptr;
  size_t cl_cap = 0;
  // cz_model_set_dictionary: every segment of cz_encode / cz_encode_dev / cz_decode is coded as if it followed these symbols
  std::vector<uint32_t> dictionary;
  // cz_model_set_match: order K of the match model (0: off); cz_model_set_match_out: per-token prediction and flag weight (match.h)
  uint32_t match_order = 0;
  uint32_t *mo_pred_host = nullptr, *mo_w_host = nullptr;
  size_t mo_cap = 0;
};

namespace cz {

int model_finalize(cz_model *m);
int ensure_workspace(cz_model *m, size_t rows, size_t n_logit, size_t n_tiles = 0);
int ensure_stage(cz_model *m, size_t bytes);
int ensure_logits(cz_model *m, size_t n_cols);
// makes `st` wait for the CDF passes still running on the side stream (their results / the logits buffers are about to be used)
int join_cdf(cz_model *m, cudaStream_t st);

// KV arena view: element (layer l, slot s) lives at base + l*layer_stride + s*kvd
struct KvView {
  __nv_bfloat16 *k = nullptr, *v = nullptr;
  size_t layer_stride = 0;  // elements
  // attention tiles (device): tile t covers rows [tile_row0[t], +tile_n[t]) = consecutive positions of one sequence,
  // starting at a position that is a multiple of 64 (or a single decode row)
  const int *tile_row0 = nullptr, *tile_n = nullptr;
  int n_tiles = 0;
  int n_slots = 0;             // valid slots of the arena (rows of k / v): TMA zero-fills beyond them
  bool single_rows = false;    // every tile is a single position (stepwise decode)
};

// embedding + all layers over n_rows rows whose metadata (tok/pos/kv_base) is already in m->ws; leaves the residual in ws.x
int forward_trunk(cz_model *m, int n_rows, const KvView &kv, cudaStream_t st);
// final RMSNorm of the n_logit rows listed in ws.logit_rows -> ws.xn_logit
int final_norm_gather(cz_model *m, int n_logit, cudaStream_t st);
// logits[V][ld] (vocab-major) for columns [col0, col0+n_cols) of ws.xn_logit
// colmax (optional, [>= n_cols] ints): receives the exact per-column max in the order-preserving int encoding; *colmax_valid
// says whether this engine produced it
int lm_head(cz_model *m, int col0, int n_cols, float *logits, size_t ld, cudaStream_t st, int *colmax = nullptr,
            bool *colmax_valid = nullptr);


// ---- f-4 logits digests (digest_kernels.cu) ----
size_t digest_scratch_bytes(size_t V, size_t n_cols);
int launch_logits_digest(cz_ctx *ctx, const float *logits, size_t V, size_t n_cols, size_t ld, void *scratch, uint8_t *out,
                         unsigned long long out_first, const unsigned long long *out_index, const uint64_t *seg_start,
                         const unsigned long long *ctr, cudaStream_t st);
// reserves the device digest buffer (n_tokens x 16 B) + hash scratch when the model has a digest sink; no-op otherwise
int digest_begin(cz_model *m, size_t n_tokens, size_t max_cols, cudaStream_t st);
// copies n_tokens digests to the sink (async on st; the caller synchronises)
int digest_end(cz_model *m, size_t n_tokens, cudaStream_t st);

// ---- RWKV-7 ----
int rwkv_finalize(cz_model *m);
void rwkv_free(cz_model *m);
int rwkv_ensure_ws(cz_model *m, size_t rows, size_t n_streams);
int rwkv_state_reset(cz_model *m, RwkvState &s, size_t n, cudaStream_t st);
void rwkv_state_free(RwkvState &s);
int rwkv_forward(cz_model *m, int n_rows, int n_streams, RwkvState &stt, bool in_place, const int *stream_active, cudaStream_t st);
int rwkv_final_norm_gather(cz_model *m, int n_logit, cudaStream_t st);

}  // namespace cz
