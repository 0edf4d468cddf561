// Model store, seeded random init, weight packing and the batched SmolLM forward (trunk + LM head).
// Replaces SmolLmSession::load (src/models.rs:48-61) and the candle Llama::forward call behind
// step_logits_tensor / reprime_with_history_and_get_last_logits_tensor (src/models.rs:92-119).
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "gemm.h"
#include "llama_kernels.h"
#include "model.h"

int GrowBuf::reserve(size_t bytes, cudaStream_t st) {
  if (bytes <= cap && p) return CZ_OK;
  if (p) {
    CZ_CUDA_TRY(cudaStreamSynchronize(st));
    cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  const size_t want = bytes + (bytes >> 3) + 256;
  CZ_CUDA_TRY(cudaMalloc(&p, want));
  cap = want;
  return CZ_OK;
}

namespace cz {

static uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
static uint64_t fnv1a64(const char *s) {
  uint64_t h = 0xcbf29ce484222325ull;
  for (; *s; s++) {
    h ^= (uint8_t)*s;
    h *= 0x100000001b3ull;
  }
  return h;
}
static uint16_t f32_to_bf16_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
static float bf16_bits_to_f32(uint16_t b) {
  uint32_t u = (uint32_t)b << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
static uint16_t f16_bits_to_bf16_bits(uint16_t h) {
  uint32_t sign = (h >> 15) & 1, e = (h >> 10) & 0x1f, mant = h & 0x3ff;
  float f;
  if (e == 0) f = ldexpf((float)mant, -24);
  else if (e == 31) f = mant ? NAN : INFINITY;
  else f = ldexpf((float)(mant | 0x400), (int)e - 25);
  return f32_to_bf16_bits(sign ? -f : f);
}

static void add_slot(cz_model *m, const std::string &name, size_t n) {
  TensorSlot s;
  s.name = name;
  s.n = n;
  m->index[name] = (int)m->tensors.size();
  m->tensors.push_back(std::move(s));
}

static int slot_of(cz_model *m, const char *name) {
  std::string key(name);
  if (key == "lm_head.weight" && m->cfg.arch == CZ_ARCH_SMOLLM) key = "model.embed_tokens.weight";  // tied head
  auto it = m->index.find(key);
  return it == m->index.end() ? -1 : it->second;
}

static bool is_norm_name(const std::string &n) { return n.find("norm") != std::string::npos; }

int upload_slot(cz_model *m, TensorSlot &s) {
  if (m->ctx->device < 0) return CZ_OK;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (!s.dev) CZ_CUDA_TRY(cudaMalloc((void **)&s.dev, s.n * 2));
  CZ_CUDA_TRY(cudaMemcpy(s.dev, s.host.data(), s.n * 2, cudaMemcpyHostToDevice));
  std::vector<uint16_t>().swap(s.host);
  return CZ_OK;
}

int ensure_stage(cz_model *m, size_t bytes) {
  Workspace &w = m->ws;
  if (bytes <= w.h_stage_bytes) return CZ_OK;
  if (w.h_stage) cudaFreeHost(w.h_stage);
  w.h_stage = nullptr;
  w.h_stage_bytes = 0;
  size_t want = bytes + (bytes >> 2) + 4096;
  CZ_CUDA_TRY(cudaMallocHost(&w.h_stage, want));
  w.h_stage_bytes = want;
  return CZ_OK;
}

template <typename T>
static int realloc_dev(T *&p, size_t n) {
  if (p) cudaFree(p);
  p = nullptr;
  if (n == 0) return CZ_OK;
  CZ_CUDA_TRY(cudaMalloc((void **)&p, n * sizeof(T)));
  return CZ_OK;
}

int ensure_workspace(cz_model *m, size_t rows, size_t n_logit, size_t n_tiles) {
  Workspace &w = m->ws;
  const cz_model_config &c = m->cfg;
  const size_t D = c.d_model, F = c.d_ffn, kvd = (size_t)c.n_kv_heads * 64, QKV = D + 2 * kvd;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (rows > w.cap_rows) {
    CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
    size_t r = rows + rows / 8 + 128;
    CZ_TRY(realloc_dev(w.x, r * D));
    CZ_TRY(realloc_dev(w.tok, r));
    if (c.arch == CZ_ARCH_RWKV7) {  // the RWKV-7 activations live in RwkvWs (rwkv7.cu)
      w.cap_rows = r;
      return ensure_workspace(m, rows, n_logit, n_tiles);
    }
    CZ_TRY(realloc_dev(w.xn, r * D));
    CZ_TRY(realloc_dev(w.ssq, r * 12));
    CZ_TRY(realloc_dev(w.qkv, r * QKV));
    CZ_TRY(realloc_dev(w.q, r * D));
    CZ_TRY(realloc_dev(w.attn, r * D));
    CZ_TRY(realloc_dev(w.act, r * F));
    CZ_TRY(realloc_dev(w.kpack, r * kvd));
    CZ_TRY(realloc_dev(w.vpack, r * kvd));
    CZ_TRY(realloc_dev(w.pos, r));
    CZ_TRY(realloc_dev(w.kv_base, r));
    w.cap_rows = r;
  }
  if (n_tiles > w.cap_tiles) {
    CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
    size_t r = n_tiles + n_tiles / 8 + 128;
    CZ_TRY(realloc_dev(w.tile_row0, r));
    CZ_TRY(realloc_dev(w.tile_n, r));
    w.cap_tiles = r;
  }
  if (n_logit > w.cap_logit) {
    CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
    size_t r = n_logit + n_logit / 8 + 128;
    CZ_TRY(realloc_dev(w.logit_rows, r));
    CZ_TRY(realloc_dev(w.syms, r));
    CZ_TRY(realloc_dev(w.out_index, r));
    CZ_TRY(realloc_dev(w.xn_logit, r * D));
    w.cap_logit = r;
  }
  return CZ_OK;
}

// Logits sub-batch buffer [V][ld_sub] (vocab-major), grow-only, sized for the widest wave seen so far: up to 262,144
// columns (51.5 GB for V = 49152).  The thread-per-column CDF kernel gets its parallelism -- and its ability to hide DRAM
// latency -- from the column count: 32,768 columns are only 7 warps per SM (measured 10% of HBM peak,
// profiles/ncu_summary_r01.md); a whole wave at once fills the SMs.
int ensure_logits(cz_model *m, size_t n_cols) {
  Workspace &w = m->ws;
  const cz_model_config &c = m->cfg;
  size_t want = (std::max<size_t>(n_cols, 256) + 1023) & ~(size_t)1023;
  // two buffers of up to sm_count x 1,024 columns (151,552 on B200: 29.8 GB each for V = 49152): wide enough for the
  // thread-per-column CDF kernels to fill the machine, and one can go through its CDF pass while the LM head fills the other.  The
  // width is two full waves of the stats kernel (256-column CTAs, two per SM): with 131,072 columns its second wave was 73% full
  // (26.8 -> 23.1 ms per bench step, profiles/ab_cols.log); halving it under memory pressure (below) leaves one full wave.
  size_t max_ld = (size_t)std::max(1, m->ctx->sm_count) * 1024;
  if (const char *e = getenv("CZ_LOGITS_COLS")) max_ld = std::max<size_t>(256, (size_t)atoll(e));
  want = std::min(want, max_ld);
  if (want <= w.ld_sub) return CZ_OK;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream2));
  w.cdf_pending[0] = w.cdf_pending[1] = false;
  CZ_TRY(realloc_dev(w.logits[0], 0));
  CZ_TRY(realloc_dev(w.logits[1], 0));
  CZ_TRY(realloc_dev(w.colmax, 0));
  w.ld_sub = 0;
  size_t free_b = 0, total_b = 0;
  CZ_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
  while (want > 256 && 2 * want * (size_t)c.vocab * 4 > free_b * 60 / 100) want >>= 1;
  CZ_TRY(realloc_dev(w.logits[0], want * (size_t)c.vocab));
  CZ_TRY(realloc_dev(w.logits[1], want * (size_t)c.vocab));
  CZ_TRY(realloc_dev(w.colmax, 2 * want));
  w.ld_sub = want;
  for (int b = 0; b < 2; b++) {
    if (!w.ev_head[b]) CZ_CUDA_TRY(cudaEventCreateWithFlags(&w.ev_head[b], cudaEventDisableTiming));
    if (!w.ev_cdf[b]) CZ_CUDA_TRY(cudaEventCreateWithFlags(&w.ev_cdf[b], cudaEventDisableTiming));
  }
  return CZ_OK;
}

int join_cdf(cz_model *m, cudaStream_t st) {
  Workspace &w = m->ws;
  for (int b = 0; b < 2; b++)
    if (w.cdf_pending[b]) {
      CZ_CUDA_TRY(cudaStreamWaitEvent(st, w.ev_cdf[b], 0));
      w.cdf_pending[b] = false;
    }
  return CZ_OK;
}

int model_finalize(cz_model *m) {
  if (m->finalized) return CZ_OK;
  if (m->ctx->device < 0) {
    set_error("model needs a GPU ctx for compute");
    return CZ_ERR_NO_DEVICE;
  }
  for (auto &s : m->tensors)
    if (!s.set) {
      set_error("tensor not set: " + s.name);
      return CZ_ERR_INVALID;
    }
  if (m->cfg.arch == CZ_ARCH_RWKV7) {
    CZ_TRY(rwkv_finalize(m));
    m->finalized = true;
    return CZ_OK;
  }
  const cz_model_config &c = m->cfg;
  const size_t D = c.d_model, F = c.d_ffn, kvd = (size_t)c.n_kv_heads * 64, QKV = D + 2 * kvd, L = c.n_layers;
  if (D % 64 || F % 64 || c.head_dim != 64 || c.n_heads * 64 != (int)D || c.n_heads % c.n_kv_heads || c.n_heads / c.n_kv_heads > 4) {
    set_error("unsupported SmolLM shape (need head_dim 64, d_model/d_ffn multiples of 64, GQA group <= 4)");
    return CZ_ERR_UNSUPPORTED;
  }
  // gate/up tile width: 256 (two 64-column chunk pairs per epilogue warp) when d_ffn allows it, else 192
  if (F % 128 == 0) m->gu_bn = 256;
  else if (F % 96 == 0) m->gu_bn = 192;
  else {
    set_error("d_ffn must be a multiple of 96 or 128");
    return CZ_ERR_UNSUPPORTED;
  }
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->w_qkv, L * QKV * D * 2));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->w_o, L * D * D * 2));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->w_gu, L * 2 * F * D * 2));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->w_d, L * D * F * 2));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->norms, (L * 2 + 1) * D * 4));
  auto dev = [&](const std::string &name) { return m->tensors[m->index[name]].dev; };
  std::vector<float> norms((L * 2 + 1) * D);
  std::vector<uint16_t> tmp(D);
  auto fetch_norm = [&](const std::string &name, float *dst) -> int {
    CZ_CUDA_TRY(cudaMemcpy(tmp.data(), dev(name), D * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < D; i++) dst[i] = bf16_bits_to_f32(tmp[i]);
    return CZ_OK;
  };
  const size_t half = m->gu_bn / 2;
  for (size_t l = 0; l < L; l++) {
    const std::string p = "model.layers." + std::to_string(l) + ".";
    __nv_bfloat16 *qkv = m->w_qkv + l * QKV * D;
    CZ_CUDA_TRY(cudaMemcpy(qkv, dev(p + "self_attn.q_proj.weight"), D * D * 2, cudaMemcpyDeviceToDevice));
    CZ_CUDA_TRY(cudaMemcpy(qkv + D * D, dev(p + "self_attn.k_proj.weight"), kvd * D * 2, cudaMemcpyDeviceToDevice));
    CZ_CUDA_TRY(cudaMemcpy(qkv + (D + kvd) * D, dev(p + "self_attn.v_proj.weight"), kvd * D * 2, cudaMemcpyDeviceToDevice));
    CZ_CUDA_TRY(cudaMemcpy(m->w_o + l * D * D, dev(p + "self_attn.o_proj.weight"), D * D * 2, cudaMemcpyDeviceToDevice));
    __nv_bfloat16 *gu = m->w_gu + l * 2 * F * D;
    // groups of `half` gate rows followed by the matching `half` up rows
    CZ_CUDA_TRY(cudaMemcpy2D(gu, 2 * half * D * 2, dev(p + "mlp.gate_proj.weight"), half * D * 2, half * D * 2, F / half,
                             cudaMemcpyDeviceToDevice));
    CZ_CUDA_TRY(cudaMemcpy2D(gu + half * D, 2 * half * D * 2, dev(p + "mlp.up_proj.weight"), half * D * 2, half * D * 2, F / half,
                             cudaMemcpyDeviceToDevice));
    CZ_CUDA_TRY(cudaMemcpy(m->w_d + l * D * F, dev(p + "mlp.down_proj.weight"), D * F * 2, cudaMemcpyDeviceToDevice));
    CZ_TRY(fetch_norm(p + "input_layernorm.weight", &norms[(l * 2) * D]));
    CZ_TRY(fetch_norm(p + "post_attention_layernorm.weight", &norms[(l * 2 + 1) * D]));
  }
  CZ_TRY(fetch_norm("model.norm.weight", &norms[L * 2 * D]));
  CZ_CUDA_TRY(cudaMemcpy(m->norms, norms.data(), norms.size() * 4, cudaMemcpyHostToDevice));
  m->embed = dev("model.embed_tokens.weight");
  m->head_w = m->embed;  // tied
  m->attn_tc = c.engine == CZ_ENGINE_TCGEN05 && getenv("CZ_ATTN_MMA") == nullptr && getenv("CZ_DEBUG_NO_FUSED_ROPE") == nullptr;
  m->attn_tile = m->attn_tc ? 128 : 64;
  // RoPE tables, same formulas as the oracle (f32 inv_freq, f32 angle, libm cosf/sinf)
  std::vector<float> ct((size_t)m->rope_max_pos * 32), stab((size_t)m->rope_max_pos * 32);
  for (int j = 0; j < 32; j++) {
    float inv_freq = 1.0f / powf(c.rope_theta, (float)(2 * j) / 64.0f);
    for (int p = 0; p < m->rope_max_pos; p++) {
      float ang = (float)p * inv_freq;
      ct[(size_t)p * 32 + j] = cosf(ang);
      stab[(size_t)p * 32 + j] = sinf(ang);
    }
  }
  CZ_CUDA_TRY(cudaMalloc((void **)&m->cos_tab, ct.size() * 4));
  CZ_CUDA_TRY(cudaMalloc((void **)&m->sin_tab, stab.size() * 4));
  CZ_CUDA_TRY(cudaMemcpy(m->cos_tab, ct.data(), ct.size() * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(m->sin_tab, stab.data(), stab.size() * 4, cudaMemcpyHostToDevice));
  m->finalized = true;
  return CZ_OK;
}

int forward_trunk(cz_model *m, int n_rows, const KvView &kv, cudaStream_t st) {
  const cz_model_config &c = m->cfg;
  cz_ctx *ctx = m->ctx;
  Workspace &w = m->ws;
  const int D = c.d_model, F = c.d_ffn, nh = c.n_heads, nkv = c.n_kv_heads, kvd = nkv * 64, QKV = D + 2 * kvd, L = c.n_layers;
  // Fused RMSNorm (tcgen05 engine): the residual-add epilogues of o_proj / down_proj (EPI_ADD_NORM) leave bf16(x * w_norm) and
  // per-row partial sums of x^2 for the norm that follows, and the consuming projection scales its accumulator rows by
  // 1/rms -- the fp32 residual is never re-read by a separate normalisation pass.  Needs D = a multiple of 192 (SmolLM-135M: 3 N tiles, n_part = 9).
  static const bool no_fused_norm = getenv("CZ_DEBUG_NO_FUSED_NORM") != nullptr;  // bisecting aid
  const bool fused_norm = c.engine == CZ_ENGINE_TCGEN05 && !no_fused_norm && getenv("CZ_DEBUG_NO_FUSED_ROPE") == nullptr && D % 192 == 0 &&
                          (D / 192) * 3 <= 12;
  // Default: the thread-per-row residual epilogue (residual in and out by TMA, one partial per N tile; 2% faster per step in
  // A/B runs); CZ_NORM_TRANSPOSE=1 selects the transposing epilogue (three warps per TMEM lane quadrant, three partials per N tile)
  static const bool norm_tma = getenv("CZ_NORM_TRANSPOSE") == nullptr;
  const int epi_norm = norm_tma ? EPI_ADD_NORM_TMA : EPI_ADD_NORM;
  const int n_part = fused_norm ? (norm_tma ? D / 192 : (D / 192) * 3) : 0;
  NormExt consume{};
  if (fused_norm) {
    consume.ssq_in = w.ssq; consume.n_part_in = n_part; consume.inv_d = 1.0f / (float)D; consume.eps = c.norm_eps;
    CZ_TRY(launch_embed_norm(ctx, m->embed, w.tok, m->norms, w.x, w.xn, w.ssq, n_rows, D, n_part, c.vocab, st));
  } else {
    CZ_TRY(launch_embed(ctx, m->embed, w.tok, w.x, n_rows, D, c.vocab, st));
  }
  for (int l = 0; l < L; l++) {
    const float *n1 = m->norms + (size_t)(2 * l) * D, *n2 = m->norms + (size_t)(2 * l + 1) * D;
    __nv_bfloat16 *kl = kv.k + (size_t)l * kv.layer_stride, *vl = kv.v + (size_t)l * kv.layer_stride;
    if (!fused_norm) CZ_TRY(launch_rmsnorm(ctx, w.x, n1, nullptr, w.xn, n_rows, D, c.norm_eps, st));
    GemmArgs g{};
    g.a = w.xn; g.lda = D; g.b = m->w_qkv + (size_t)l * QKV * D; g.ldb = D; g.c = w.qkv; g.ldc = QKV;
    g.M = n_rows; g.N = QKV; g.K = D; g.epi = EPI_STORE_F32; g.bn = 192; g.fam = CZ_K_GEMM;
    static const bool no_fused_rope = getenv("CZ_DEBUG_NO_FUSED_ROPE") != nullptr;  // bisecting aid
    if (c.engine == CZ_ENGINE_TCGEN05 && !no_fused_rope) {
      // RoPE + bf16 conversion + K/V arena scatter fused into the projection's epilogue: the fp32 qkv rows never reach HBM
      g.epi = EPI_QKV_ROPE;
      g.c = nullptr;
      g.rope.pos = w.pos; g.rope.kv_base = w.kv_base; g.rope.cos_tab = m->cos_tab; g.rope.sin_tab = m->sin_tab;
      g.rope.q = w.q; g.rope.k_arena = kl; g.rope.nh = nh; g.rope.nkv = nkv;
      g.rope.v_arena = vl;  // V rows [slot][nkv*64] for both attention kernels (the tcgen05 one reads them as an MN-major operand)
      if (fused_norm) g.norm = consume;
      CZ_TRY(gemm(ctx, c.engine, g, st));
      g.rope = RopeExt();
      g.norm = NormExt();
    } else {
      CZ_TRY(gemm(ctx, c.engine, g, st));
      CZ_TRY(launch_rope_split(ctx, w.qkv, w.pos, w.kv_base, m->cos_tab, m->sin_tab, w.q, kl, vl, n_rows, nh, nkv, st));
    }
    static const bool force_rows = getenv("CZ_DEBUG_ATTN_ROWS") != nullptr;  // bisecting aid
    if (m->attn_tc)
      CZ_TRY(launch_attn_tc(ctx, w.q, n_rows, kl, vl, kv.n_slots, 0, w.pos, w.kv_base, kv.tile_row0,
                            kv.tile_n, kv.n_tiles, w.attn, nh, nkv, kv.single_rows, st));
    else if (c.engine == CZ_ENGINE_TCGEN05 && !force_rows)
      CZ_TRY(launch_attn_mma(ctx, w.q, kl, vl, w.pos, w.kv_base, kv.tile_row0, kv.tile_n, kv.n_tiles, w.attn, nh, nkv, st));
    else
      CZ_TRY(launch_attn_rows(ctx, w.q, kl, vl, w.pos, w.kv_base, w.attn, n_rows, nh, nkv, st));
    g.a = w.attn; g.lda = D; g.b = m->w_o + (size_t)l * D * D; g.ldb = D; g.c = w.x; g.ldc = D;
    g.M = n_rows; g.N = D; g.K = D; g.epi = EPI_ADD_F32; g.bn = 192; g.fam = CZ_K_GEMM_O;
    if (fused_norm) {  // x += attn * Wo^T, and the FFN norm's inputs
      g.epi = epi_norm;
      g.norm.w_next = n2; g.norm.xb = w.xn; g.norm.ssq_out = w.ssq;
    }
    CZ_TRY(gemm(ctx, c.engine, g, st));
    g.norm = NormExt();
    if (!fused_norm) CZ_TRY(launch_rmsnorm(ctx, w.x, n2, nullptr, w.xn, n_rows, D, c.norm_eps, st));
    g.a = w.xn; g.lda = D; g.b = m->w_gu + (size_t)l * 2 * F * D; g.ldb = D; g.c = w.act; g.ldc = F;
    g.M = n_rows; g.N = 2 * F; g.K = D; g.epi = EPI_SWIGLU_BF16; g.bn = m->gu_bn; g.fam = CZ_K_GEMM_GU;
    if (fused_norm) g.norm = consume;
    CZ_TRY(gemm(ctx, c.engine, g, st));
    g.norm = NormExt();
    g.a = w.act; g.lda = F; g.b = m->w_d + (size_t)l * D * F; g.ldb = F; g.c = w.x; g.ldc = D;
    g.M = n_rows; g.N = D; g.K = F; g.epi = EPI_ADD_F32; g.bn = 192; g.fam = CZ_K_GEMM_DOWN;
    if (fused_norm && l + 1 < L) {  // x += act * Wd^T, and the next layer's attention norm's inputs (the final norm reads fp32 x)
      g.epi = epi_norm;
      g.norm.w_next = m->norms + (size_t)(2 * (l + 1)) * D; g.norm.xb = w.xn; g.norm.ssq_out = w.ssq;
    }
    CZ_TRY(gemm(ctx, c.engine, g, st));
    g.norm = NormExt();
  }
  return CZ_OK;
}

int final_norm_gather(cz_model *m, int n_logit, cudaStream_t st) {
  const cz_model_config &c = m->cfg;
  return launch_rmsnorm(m->ctx, m->ws.x, m->norms + (size_t)(2 * c.n_layers) * c.d_model, m->ws.logit_rows, m->ws.xn_logit,
                        n_logit, c.d_model, c.norm_eps, st);
}

int launch_fill_i32(cz_ctx *ctx, int *p, int v, size_t n, cudaStream_t stream);

int lm_head(cz_model *m, int col0, int n_cols, float *logits, size_t ld, cudaStream_t st, int *colmax, bool *colmax_valid) {
  const cz_model_config &c = m->cfg;
  static const bool no_colmax = getenv("CZ_DEBUG_NO_COLMAX") != nullptr;  // bisecting aid
  const bool fuse_max = colmax && c.engine == CZ_ENGINE_TCGEN05 && !no_colmax;
  if (colmax_valid) *colmax_valid = fuse_max;
  if (fuse_max) CZ_TRY(launch_fill_i32(m->ctx, colmax, INT_MIN, (size_t)n_cols, st));
  GemmArgs g{};
  g.a = m->head_w; g.lda = c.d_model;                      // A = LM head [V][D] (SmolLM: the tied embedding): vocab is the M dimension
  g.b = m->ws.xn_logit + (size_t)col0 * c.d_model; g.ldb = c.d_model;  // B = hidden states: tokens are the N dimension
  g.c = logits; g.ldc = (int)ld;                           // -> vocab-major logits [V][ld]
  g.M = c.vocab; g.N = n_cols; g.K = c.d_model; g.epi = fuse_max ? EPI_STORE_F32_COLMAX : EPI_STORE_F32; g.bn = 256;
  g.aux = colmax;
  g.fam = CZ_K_GEMM_HEAD;
  return gemm(m->ctx, c.engine, g, st);
}

}  // namespace cz

using namespace cz;

extern "C" {

void cz_model_config_smollm_135m(cz_model_config *cfg) {
  memset(cfg, 0, sizeof(*cfg));
  cfg->arch = CZ_ARCH_SMOLLM;
  cfg->vocab = 49152;
  cfg->d_model = 576;
  cfg->n_layers = 30;
  cfg->n_heads = 9;
  cfg->n_kv_heads = 3;
  cfg->head_dim = 64;
  cfg->d_ffn = 1536;
  cfg->norm_eps = 1e-5f;
  cfg->rope_theta = 100000.0f;
  cfg->engine = CZ_ENGINE_TCGEN05;
}
void cz_model_config_rwkv7_0p1b(cz_model_config *cfg) {
  memset(cfg, 0, sizeof(*cfg));
  cfg->arch = CZ_ARCH_RWKV7;
  cfg->vocab = 65536;
  cfg->d_model = 768;
  cfg->n_layers = 12;
  cfg->n_heads = 12;
  cfg->head_dim = 64;
  cfg->d_ffn = 3072;
  cfg->norm_eps = 1e-5f;
  cfg->lora_w = 64;
  cfg->lora_a = 64;
  cfg->lora_v = 32;
  cfg->lora_g = 128;
  cfg->engine = CZ_ENGINE_TCGEN05;
}

int cz_model_create(cz_ctx *ctx, const cz_model_config *cfg, cz_model **out) {
  if (!ctx || !cfg || !out) return CZ_ERR_INVALID;
  cz_model *m = new cz_model();
  m->ctx = ctx;
  m->cfg = *cfg;
  const size_t D = cfg->d_model, F = cfg->d_ffn, V = cfg->vocab;
  if (cfg->arch == CZ_ARCH_SMOLLM) {
    const size_t kvd = (size_t)cfg->n_kv_heads * cfg->head_dim;
    add_slot(m, "model.embed_tokens.weight", V * D);
    for (int l = 0; l < cfg->n_layers; l++) {
      const std::string p = "model.layers." + std::to_string(l) + ".";
      add_slot(m, p + "input_layernorm.weight", D);
      add_slot(m, p + "self_attn.q_proj.weight", D * D);
      add_slot(m, p + "self_attn.k_proj.weight", kvd * D);
      add_slot(m, p + "self_attn.v_proj.weight", kvd * D);
      add_slot(m, p + "self_attn.o_proj.weight", D * D);
      add_slot(m, p + "post_attention_layernorm.weight", D);
      add_slot(m, p + "mlp.gate_proj.weight", F * D);
      add_slot(m, p + "mlp.up_proj.weight", F * D);
      add_slot(m, p + "mlp.down_proj.weight", D * F);
    }
    add_slot(m, "model.norm.weight", D);
  } else if (cfg->arch == CZ_ARCH_RWKV7) {
    // tensor names follow candle_rwkv7/convert_pth_direct.py:11-134 (loader: rwkv7.rs:105-144, 404-409, 443-506)
    add_slot(m, "model.embeddings.weight", V * D);
    for (int l = 0; l < cfg->n_layers; l++) {
      const std::string p = "model.layers." + std::to_string(l) + ".";
      if (l == 0) {
        add_slot(m, p + "pre_norm.weight", D);
        add_slot(m, p + "pre_norm.bias", D);
      }
      for (const char *nm : {"attn_norm", "ffn_norm"}) {
        add_slot(m, p + nm + ".weight", D);
        add_slot(m, p + nm + ".bias", D);
      }
      const std::string a = p + "attn.";
      for (const char *nm : {"r_proj", "k_proj", "v_proj", "o_proj"}) add_slot(m, a + nm + ".weight", D * D);
      add_slot(m, a + "g_norm.weight", D);
      add_slot(m, a + "g_norm.bias", D);
      for (const char *nm : {"x_r", "x_w", "x_k", "x_v", "x_a", "x_g", "k_k", "k_a", "r_k"}) add_slot(m, a + nm, D);
      add_slot(m, a + "w_lora.lora.0.weight", (size_t)cfg->lora_w * D);
      add_slot(m, a + "w_lora.lora.2.weight", D * cfg->lora_w);
      add_slot(m, a + "w_lora.lora.2.bias", D);
      add_slot(m, a + "a_lora.lora.0.weight", (size_t)cfg->lora_a * D);
      add_slot(m, a + "a_lora.lora.2.weight", D * cfg->lora_a);
      add_slot(m, a + "a_lora.lora.2.bias", D);
      if (l > 0) {
        add_slot(m, a + "v_lora.lora.0.weight", (size_t)cfg->lora_v * D);
        add_slot(m, a + "v_lora.lora.2.weight", D * cfg->lora_v);
        add_slot(m, a + "v_lora.lora.2.bias", D);
      }
      add_slot(m, a + "g_lora.lora.0.weight", (size_t)cfg->lora_g * D);
      add_slot(m, a + "g_lora.lora.2.weight", D * cfg->lora_g);
      add_slot(m, p + "ffn.x_k", D);
      add_slot(m, p + "ffn.key.weight", F * D);
      add_slot(m, p + "ffn.value.weight", D * F);
    }
    add_slot(m, "model.norm.weight", D);
    add_slot(m, "model.norm.bias", D);
    add_slot(m, "lm_head.weight", V * D);
  } else {
    delete m;
    set_error("unknown arch");
    return CZ_ERR_INVALID;
  }
  *out = m;
  return CZ_OK;
}

void cz_model_free(cz_model *m) {
  if (!m) return;
  if (m->ctx->device >= 0) {
    cudaSetDevice(m->ctx->device);
    cudaDeviceSynchronize();
    for (auto &s : m->tensors)
      if (s.dev) cudaFree(s.dev);
    for (auto &b : m->sb)
      if (b.p) cudaFree(b.p);
    void *ptrs[] = {m->w_qkv, m->w_o, m->w_gu, m->w_d, m->norms, m->cos_tab, m->sin_tab, m->ws.x, m->ws.xn, m->ws.qkv, m->ws.q,
                    m->ws.attn, m->ws.act, m->ws.kpack, m->ws.vpack, m->ws.tok, m->ws.pos, m->ws.kv_base, m->ws.logit_rows,
                    m->ws.syms, m->ws.out_index, m->ws.tile_row0, m->ws.tile_n, m->ws.xn_logit, m->ws.lo_tmp, m->ws.hi_tmp, m->ws.xe_tmp, m->ws.colmax, m->ws.logits[0],
                    m->ws.logits[1]};
    for (void *p : ptrs)
      if (p) cudaFree(p);
    if (m->ws.h_stage) cudaFreeHost(m->ws.h_stage);
    rwkv_free(m);
  }
  delete m;
}

int cz_model_config_get(const cz_model *m, cz_model_config *out) {
  if (!m || !out) return CZ_ERR_INVALID;
  *out = m->cfg;
  return CZ_OK;
}
int cz_model_set_pdf_floor(cz_model *m, int enabled) {
  if (!m) return CZ_ERR_INVALID;
  if (enabled && m->cfg.arch != CZ_ARCH_SMOLLM) {
    set_error("pdf floor: only the SmolLM alphabet has an unfloored pdf (RWKV-7 codes with a floor already)");
    return CZ_ERR_UNSUPPORTED;
  }
  m->pdf_floor = enabled != 0;
  return CZ_OK;
}
int cz_model_set_zero_width_out(cz_model *m, uint64_t *first_zw_out, size_t cap_segments) {
  if (!m || (first_zw_out && cap_segments == 0)) return CZ_ERR_INVALID;
  m->zw_host = first_zw_out;
  m->zw_cap = first_zw_out ? cap_segments : 0;
  return CZ_OK;
}
int cz_model_tensor_count(const cz_model *m) { return m ? (int)m->tensors.size() : 0; }
int cz_model_tensor_info(const cz_model *m, int idx, const char **name, size_t *n_elems) {
  if (!m || idx < 0 || idx >= (int)m->tensors.size()) return CZ_ERR_INVALID;
  if (name) *name = m->tensors[idx].name.c_str();
  if (n_elems) *n_elems = m->tensors[idx].n;
  return CZ_OK;
}

int cz_model_set_tensor(cz_model *m, const char *name, const void *data, int dtype, size_t n_elems) {
  if (!m || !name || !data) return CZ_ERR_INVALID;
  int si = slot_of(m, name);
  if (si < 0) {
    set_error(std::string("unknown tensor name: ") + name);
    return CZ_ERR_INVALID;
  }
  TensorSlot &s = m->tensors[si];
  if (s.n != n_elems) {
    set_error(std::string("size mismatch for ") + name + ": want " + std::to_string(s.n) + " got " + std::to_string(n_elems));
    return CZ_ERR_INVALID;
  }
  if (m->finalized) {
    set_error("model already finalized (weights are packed on first use)");
    return CZ_ERR_INVALID;
  }
  s.host.resize(n_elems);
  if (dtype == CZ_DTYPE_F32) {
    const float *f = (const float *)data;
    for (size_t i = 0; i < n_elems; i++) s.host[i] = f32_to_bf16_bits(f[i]);
  } else if (dtype == CZ_DTYPE_BF16) {
    memcpy(s.host.data(), data, n_elems * 2);
  } else if (dtype == CZ_DTYPE_F16) {
    const uint16_t *h = (const uint16_t *)data;
    for (size_t i = 0; i < n_elems; i++) s.host[i] = f16_bits_to_bf16_bits(h[i]);
  } else {
    set_error("unknown dtype");
    return CZ_ERR_INVALID;
  }
  s.set = true;
  return upload_slot(m, s);
}

int cz_model_get_tensor(cz_model *m, const char *name, float *out, size_t n_elems) {
  if (!m || !name || !out) return CZ_ERR_INVALID;
  int si = slot_of(m, name);
  if (si < 0 || m->tensors[si].n != n_elems || !m->tensors[si].set) {
    set_error(std::string("get_tensor: unknown / unset / size mismatch: ") + name);
    return CZ_ERR_INVALID;
  }
  TensorSlot &s = m->tensors[si];
  std::vector<uint16_t> tmp;
  const uint16_t *src;
  if (s.dev) {
    tmp.resize(n_elems);
    CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
    CZ_CUDA_TRY(cudaMemcpy(tmp.data(), s.dev, n_elems * 2, cudaMemcpyDeviceToHost));
    src = tmp.data();
  } else {
    src = s.host.data();
  }
  for (size_t i = 0; i < n_elems; i++) out[i] = bf16_bits_to_f32(src[i]);
  return CZ_OK;
}

int cz_model_random_init(cz_model *m, uint64_t seed, float std, float embed_std) {
  if (!m) return CZ_ERR_INVALID;
  if (m->finalized) {
    set_error("model already finalized");
    return CZ_ERR_INVALID;
  }
  for (auto &s : m->tensors) {
    s.host.resize(s.n);
    const bool norm_w = is_norm_name(s.name) && s.name.find("weight") != std::string::npos;
    const bool bias = s.name.size() > 5 && s.name.compare(s.name.size() - 5, 5, ".bias") == 0;
    const bool emb = s.name.find("embed") != std::string::npos || s.name == "lm_head.weight";
    if (norm_w) {
      for (size_t i = 0; i < s.n; i++) s.host[i] = 0x3f80;  // 1.0
    } else if (bias && is_norm_name(s.name)) {
      for (size_t i = 0; i < s.n; i++) s.host[i] = 0;
    } else {
      const float sd = emb ? embed_std : std;
      const float k = sd * 1.7320508075688772f / 65536.0f;
      const uint64_t ts = splitmix64(seed ^ fnv1a64(s.name.c_str()));
      for (size_t i = 0; i < s.n; i++) {
        uint64_t h = splitmix64(ts + (uint64_t)i * 0x9E3779B97F4A7C15ull);
        int sum = (int)(h & 0xFFFF) + (int)((h >> 16) & 0xFFFF) + (int)((h >> 32) & 0xFFFF) + (int)((h >> 48) & 0xFFFF);
        s.host[i] = f32_to_bf16_bits((float)(sum - 131070) * k);
      }
    }
    s.set = true;
    CZ_TRY(upload_slot(m, s));
  }
  return CZ_OK;
}

}  // extern "C"
