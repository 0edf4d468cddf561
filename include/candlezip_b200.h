/*
 * candlezip_b200.h -- C ABI of libcandlezip_b200.so: the B200-native replacement for CandleZip's
 * model-driven entropy-coding hot path.  Plain pointers and sizes only; no torch / C++ types.
 *
 * Reference interface replaced (all citations relative to the reference repo turtle261/candlezip):
 *   trait LanguageModelSession                src/models.rs:28-33      -> cz_session_*  (batch-of-1 shim)
 *   SmolLmSession::{load,index_pos,step,..}   src/models.rs:48-119     -> cz_model_* + cz_session_*
 *   softmax_pdf + quantize_pdf_to_cdf         src/main.rs:784-824      -> cz_cdf_bounds / cz_cdf_search
 *   softmax_pdf_floor / combined_pdf_with_..  src/main.rs:758-782      -> mode CZ_CDF_RWKV_LITERALS / cz_xe_*
 *   ArithmeticEncoder / ArithmeticDecoder     src/main.rs:261-549      -> cz_ac_encode_lanes / cz_ac_decode_lanes
 *   encode loop + reprime schedule            src/main.rs:1913-2358    -> cz_encode
 *   decode loop                               src/main.rs:2485-2654    -> cz_decode
 *   cross_entropy_bits_over_span              src/main.rs:1725-1787    -> cz_xe_bits
 *   container v2 (+ segment extension)        src/main.rs:227-259,551-677 -> cz_container_*
 *
 * Conventions: every function returns CZ_OK (0) or a negative cz_status; nothing throws or aborts
 * across the boundary; cz_last_error() gives a human-readable message for the last failure on the
 * calling thread.  All buffers are caller-allocated HOST memory unless the name ends in _dev.
 * One host thread per cz_ctx; a ctx owns exactly one GPU (one process per GPU, SURVEY 8e).
 * There is NO CPU fallback: without a usable sm_100 device every compute entry point fails with
 * CZ_ERR_NO_DEVICE.
 */
#ifndef CANDLEZIP_B200_H
#define CANDLEZIP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CZ_ABI_VERSION 1
#define CZ_AC_CDF_TOTAL (1u << 30) /* src/main.rs:803 */

typedef enum {
  CZ_OK = 0,
  CZ_ERR_INVALID = -1,      /* bad argument */
  CZ_ERR_NO_DEVICE = -2,    /* no CUDA device / not sm_100 */
  CZ_ERR_CUDA = -3,         /* CUDA runtime failure (message has the detail) */
  CZ_ERR_ZERO_WIDTH = -4,   /* a coded symbol has c_lo == c_hi: the reference would corrupt the stream (SURVEY 7.3a) */
  CZ_ERR_FORMAT = -5,       /* container parse error */
  CZ_ERR_NOMEM = -6,
  CZ_ERR_UNSUPPORTED = -7,
  CZ_ERR_SYMBOL_RANGE = -8, /* symbol id >= number of coded symbols */
  CZ_ERR_IO = -9
} cz_status;

typedef struct cz_ctx cz_ctx;
typedef struct cz_model cz_model;
typedef struct cz_session cz_session;

/* ---------------------------------------------------------------- context */
int cz_abi_version(void);
int cz_init(int device_id, cz_ctx **out);
void cz_shutdown(cz_ctx *ctx);
const char *cz_last_error(void);
/* number of kernel launches issued by this ctx since creation (bench.py's gpu_launches) */
uint64_t cz_launch_count(const cz_ctx *ctx);
/* per-kernel-family device time accounting (CUDA events on the ctx stream); family ids below.
 * enable, run, then read accumulated milliseconds + launches. */
enum {
  CZ_K_GEMM = 0, /* qkv projection (and generic GEMM calls) */
  CZ_K_ATTN = 1, CZ_K_ELEMWISE = 2, CZ_K_CDF = 3, CZ_K_CODER = 4, CZ_K_OTHER = 5,
  CZ_K_GEMM_O = 6, CZ_K_GEMM_GU = 7, CZ_K_GEMM_DOWN = 8, CZ_K_GEMM_HEAD = 9,
  CZ_K_CDF_PREFIX = 10, /* the encode-side prefix walk (CZ_K_CDF keeps the full passes and the decode-side search) */
  CZ_K_FAMILIES = 11
};
/* mode 0 off; 1 synchronous (sync after every launch: exact per-launch times, perturbs the step); 2 deferred
 * (event pairs recorded around every launch, read back in cz_profile_read: does not perturb the timed region) */
int cz_profile_enable(cz_ctx *ctx, int mode);
/* the cudaStream_t every kernel of this ctx is launched on (so callers can bracket work with their own events) */
void *cz_ctx_stream(cz_ctx *ctx);
int cz_profile_read(cz_ctx *ctx, double ms_out[CZ_K_FAMILIES], uint64_t launches_out[CZ_K_FAMILIES], int reset);

/* ---------------------------------------------------------------- K1: logits -> integer CDF */
enum {
  CZ_CDF_SMOLLM = 0,        /* softmax_pdf, no floor: src/main.rs:2294-2296 */
  CZ_CDF_RWKV_LITERALS = 1, /* floor 2^-29, 256 literal symbols appended: src/main.rs:2303-2321 */
  CZ_CDF_SMOLLM_FLOOR = 2   /* quantize_pdf_to_cdf(softmax_pdf_floor(logits, 2^-29)) over the V vocabulary symbols (src/main.rs:758-767):
                               the SmolLM alphabet with the floor the reference's RWKV coder and gate XE use.  No symbol is ever
                               zero-width: with f = 2^-29, p_i = max(e_i / S, f) / norm and norm <= 1 + V f (+ rounding), p_i 2^30 >=
                               2 / norm > 1 whenever V < 2^29, so consecutive partial sums differ by more than one quantum and every
                               cdf[i+1] - cdf[i] >= 1 (no partial sum before the last reaches 1; the clamp at 2^30 only touches
                               cdf[V]).  For cz_xe_bits_cols the mode is the same as CZ_CDF_SMOLLM (which already floors there). */
};
/* logits are VOCAB-MAJOR: logits[v * ld + m], m = 0..M-1 (one column per stream/token), ld >= M.
 * For each column m: (c_lo, c_hi) = (cdf[sym], cdf[sym+1]) of the reference's quantised CDF, bit-exact.
 * c_lo == c_hi is reported per column (not an error here); cz_encode turns it into CZ_ERR_ZERO_WIDTH. */
int cz_cdf_bounds(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode,
                  const uint32_t *syms, uint32_t *c_lo, uint32_t *c_hi);
int cz_cdf_bounds_dev(cz_ctx *ctx, const float *logits_dev, size_t vocab, size_t m, size_t ld, int mode,
                      const uint32_t *syms_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev);
/* decode side: for each column the symbol s with cdf[s] <= value < cdf[s+1] (src/main.rs:507-516) and its bounds */
int cz_cdf_search(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode,
                  const uint32_t *values, uint32_t *syms_out, uint32_t *c_lo, uint32_t *c_hi);
/* full CDF of ONE column (vocab+1 or vocab+257 entries) -- debugging / watchdog parity, not a hot path */
int cz_cdf_full(cz_ctx *ctx, const float *logits, size_t vocab, int mode, uint32_t *cdf_out);
/* K9: -log2(max(p_floor(sym), 1e-300)) per column (src/main.rs:1745-1747 / 1778-1781) */
int cz_xe_bits_cols(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode,
                    const uint32_t *syms, double *bits_out);
/* Expected code length, in bits, of each column's coding distribution in `mode` (0, 1 or 2; else CZ_ERR_INVALID):
 *   bits_out[m] = 2^-30 * sum_{s < n, w_s > 0} w_s * (30 - log2 w_s),   w_s = cdf[s+1] - cdf[s]
 * with cdf[0..n] exactly the quantised CDF the coder uses (cz_cdf_full's; n = vocab, or vocab + 256 with CZ_CDF_RWKV_LITERALS),
 * summed in f64 in ascending s by one thread per column: a pure function of the column, whatever the batch.  Arguments as cz_cdf_bounds. */
int cz_cdf_entropy(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode, double *bits_out);

/* ---------------------------------------------------------------- K2/K3: arithmetic coder lanes */
/* Lane l codes the interval list [lane_off[l], lane_off[l+1]) of (c_lo, c_hi) with total 2^30, then finish().
 * out_off[l] (in/out): on input the byte offset of lane l's output region inside `out` (regions must be
 * >= 4*(n_l)+8 bytes); out_len[l] receives the payload length.  Bit-exact with src/main.rs:353-399. */
int cz_ac_encode_lanes(cz_ctx *ctx, const uint32_t *c_lo, const uint32_t *c_hi, const uint64_t *lane_off,
                       size_t n_lanes, uint8_t *out, const uint64_t *out_off, uint64_t *out_len);
/* Static-model decode of lanes (test / KAT entry point): every lane uses the same CDF table `cdf`
 * (n_sym+1 entries).  payload regions as above.  syms_out laid out like the encoder's interval list. */
int cz_ac_decode_lanes(cz_ctx *ctx, const uint8_t *payload, const uint64_t *pay_off, const uint64_t *pay_len,
                       const uint64_t *lane_off, size_t n_lanes, const uint32_t *cdf, size_t n_sym,
                       uint32_t *syms_out);

/* ---------------------------------------------------------------- models */
enum { CZ_ARCH_SMOLLM = 0, CZ_ARCH_RWKV7 = 1 };
enum { CZ_DTYPE_F32 = 0, CZ_DTYPE_BF16 = 1, CZ_DTYPE_F16 = 2 };
/* which kernels compute the dense contractions; recorded in the segment extension so a stream is
 * always decoded with the arithmetic it was encoded with */
enum { CZ_ENGINE_TCGEN05 = 0, CZ_ENGINE_SIMT = 1 };

typedef struct {
  int arch;        /* CZ_ARCH_* */
  int vocab;
  int d_model;
  int n_layers;
  int n_heads;     /* smollm: query heads; rwkv7: d_model / head_dim */
  int n_kv_heads;  /* smollm only */
  int head_dim;    /* 64 */
  int d_ffn;
  float norm_eps;  /* smollm rms_norm_eps 1e-5; rwkv7 layer-norm eps 1e-5 */
  float rope_theta;
  int lora_w, lora_a, lora_v, lora_g; /* rwkv7 low-rank dims (64/64/32/128) */
  int engine;      /* CZ_ENGINE_* */
} cz_model_config;

/* SmolLM2-135M (vocab 49152, d 576, 30 layers, 9q/3kv heads, ffn 1536, theta 1e5) */
void cz_model_config_smollm_135m(cz_model_config *cfg);
/* rwkv7-g1-0.1b (vocab 65536, d 768, 12 layers, head 64, ffn 3072) */
void cz_model_config_rwkv7_0p1b(cz_model_config *cfg);

int cz_model_create(cz_ctx *ctx, const cz_model_config *cfg, cz_model **out);
void cz_model_free(cz_model *m);
/* HF tensor names ("model.layers.3.self_attn.q_proj.weight", ...). Stored as bf16 on device (SmolLM2 ships bf16). */
int cz_model_set_tensor(cz_model *m, const char *name, const void *data, int dtype, size_t n_elems);
/* read a tensor back as f32 exactly as the kernels see it (tests hand these to the oracle) */
int cz_model_get_tensor(cz_model *m, const char *name, float *out, size_t n_elems);
/* number of tensors + their names/sizes, for enumeration */
int cz_model_tensor_count(const cz_model *m);
int cz_model_tensor_info(const cz_model *m, int idx, const char **name, size_t *n_elems);
/* seeded random-init weights of the same architecture (no checkpoints offline): counter-based hash,
 * ~N(0, std) as a sum of 4 uniforms, norm weights = 1, values rounded to bf16. `embed_std` lets a test
 * make the logits peaky. Usable without a GPU when m was created on a ctx opened with device_id = -1. */
int cz_model_random_init(cz_model *m, uint64_t seed, float std, float embed_std);
/* minimal safetensors reader (F32 / BF16 / F16), HF LLaMA or candle_rwkv7 tensor names */
int cz_model_load_safetensors(cz_model *m, const char *const *paths, int n_paths);
int cz_model_config_get(const cz_model *m, cz_model_config *out);

/* ---------------------------------------------------------------- LanguageModelSession shim (batch of 1) */
int cz_session_new(cz_model *m, cz_session **out);
void cz_session_free(cz_session *s);
size_t cz_session_vocab_size(const cz_session *s);
size_t cz_session_max_context_length(const cz_session *s); /* 512 for smollm (src/models.rs:91) */
size_t cz_session_index_pos(const cz_session *s);
int cz_session_step_logits(cz_session *s, uint32_t token, float *logits_out /* [vocab] */);
int cz_session_reprime(cz_session *s, const uint32_t *history, size_t n, float *logits_out);

/* ---------------------------------------------------------------- batched hot path */
typedef struct {
  uint64_t i;                /* loop index at which the prime is applied (i + 1 == agent boundary) */
  const uint32_t *prime;     /* explicit tokens fed after the history tail: hint[..budget] (src/main.rs:2123-2146) */
  uint32_t prime_len;
  uint64_t hold_until;       /* src/main.rs:2149 */
  uint32_t hist_take;        /* tokens taken from the stream itself before `prime`: tail(ids[..=i], hist_take) with ids[0] = BOS
                                (src/main.rs:2132-2134, 2596-2600).  The decoder rebuilds this part from what it has decoded, so a
                                gated stream decodes in one call.  0: `prime` is the whole prime.  RWKV-7: the last hist_take
                                symbols below vocab before index i (literal escapes skipped), BOS first when there are fewer. */
} cz_prime_event;

typedef struct {
  uint32_t context;          /* --context (512) */
  uint32_t reprime_interval; /* --reprime-interval (512) */
  uint32_t n_segments;       /* independently-coded segments; 1 == the reference's single stream */
  const uint64_t *seg_start; /* [n_segments+1] offsets into the CODED token list ids[1..]; seg_start[0]=0, last=n_tokens */
  uint32_t bos;
  const cz_prime_event *events; /* only valid with n_segments == 1; may be NULL */
  uint32_t n_events;
  uint32_t max_batch_tokens; /* teacher-forced rows per wave (0 = default) */
} cz_schedule;

typedef struct {
  uint8_t *data;             /* caller-allocated, capacity cap */
  size_t cap;
  uint64_t *seg_off;         /* [n_segments+1] filled: payload of segment g is data[seg_off[g] .. seg_off[g+1]) */
} cz_bitstreams;

/* coded tokens: ids[0..n_tokens) (BOS is NOT included; every segment is started from sched->bos).
 * Every id is validated against the coded alphabet (vocab; vocab + 256 with RWKV-7's literal escapes) before anything is launched:
 * CZ_ERR_SYMBOL_RANGE names the offending index.  sched->bos and the hint-prime tokens are validated the same way. */
int cz_encode(cz_model *m, const uint32_t *ids, size_t n_tokens, const cz_schedule *sched, cz_bitstreams *out);
/* Lock-step batched decoder: all segments advance one token per step, column g of the logits batch being segment g.
 * PRECONDITION: segment lengths must be NON-INCREASING (longest first; cz_schedule.seg_start as produced by an even split with
 * the remainder on the first segments) so that the live streams are always a prefix of the batch; otherwise CZ_ERR_UNSUPPORTED.
 * Memory: the KV arenas are allocated up front, 2 * n_layers * n_segments * max_pos * n_kv_heads * 64 bf16 elements with
 * max_pos = 1024 at --context 512 / --reprime-interval 512 (SmolLM-135M: 23.6 MB per segment, 48 GB at 2048 segments);
 * CZ_ERR_CUDA (out of memory) if that does not fit.
 * Hint-prime events (n_segments == 1) are applied at the same coded index as cz_encode applies them, on both backends; an event's
 * history tail (hist_take) is rebuilt from the symbols decoded so far.  RWKV-7 feeds a prime in slabs of at most max_batch_tokens
 * rows (262,144 when 0), so its memory does not grow with the history; an event whose prime has no in-vocabulary token is
 * CZ_ERR_INVALID, as in cz_encode. */
int cz_decode(cz_model *m, const uint8_t *payload, const uint64_t *seg_off, size_t n_tokens,
              const cz_schedule *sched, uint32_t *ids_out);
/* device-resident variant of the encode step used by bench.py for the kernel-only number: ids already in HBM (an id outside
 * the coded alphabet is caught on the device: the call returns CZ_ERR_SYMBOL_RANGE and nothing is read out of bounds) */
int cz_encode_dev(cz_model *m, const uint32_t *ids_dev, size_t n_tokens, const cz_schedule *sched,
                  uint8_t *out_dev, size_t out_cap, uint64_t *seg_off_host);

/* f-4 watchdog digests: blake3_f32_bin16 (src/main.rs:955-961; enabled there by CANDLEZIP_WATCHDOG_DIGEST, :1085-1090; one
 * `pdf_digest` per encode / decode step, :2328-2342, :2629-2647).  With a sink set, cz_encode / cz_encode_dev / cz_decode hash
 * every coded token's logits vector (the V f32 values, little-endian) ON THE DEVICE next to the CDF pass and copy the 16-byte
 * BLAKE3-128 digests to digests_out[i * 16 .. i * 16 + 16), i = global coded index.  Encode and decode digests of a stream are
 * equal byte for byte (decode safety), whatever the wave size, batch size or GPU count.  NULL disables.  Both backends; on RWKV-7 a
 * literal-escape symbol does not step the model, so its digest is that of the logits the previous symbol was coded from. */
int cz_model_set_digest_out(cz_model *m, uint8_t *digests_out, size_t cap_tokens);

/* enabled != 0: cz_encode / cz_encode_dev / cz_decode code SmolLM streams with CZ_CDF_SMOLLM_FLOOR instead of CZ_CDF_SMOLLM, so no
 * token can be zero-width (CZ_ERR_ZERO_WIDTH cannot occur); the stream must be decoded with the same setting (the container's
 * CZ_FLAG_PDF_FLOOR).  cz_xe_bits, the session shim and cz_chunk_logits are unaffected.  Off when the model is created.
 * RWKV-7: enabled != 0 returns CZ_ERR_UNSUPPORTED (its alphabet is floored already). */
int cz_model_set_pdf_floor(cz_model *m, int enabled);

/* Per-segment zero-width report.  With a sink set, cz_encode / cz_encode_dev do not fail on a zero-width interval (SmolLM's unfloored
 * pdf, CZ_ERR_ZERO_WIDTH): they return CZ_OK and write first_zw_out[g] for every segment g of the call, the SEGMENT-RELATIVE coded
 * index of segment g's first zero-width token (the arithmetic-coder lane stops there), or UINT64_MAX when the segment has none.
 * The payload of a segment with an entry other than UINT64_MAX is UNSPECIFIED (the caller stores or re-codes that data); every other
 * segment's payload is the one it gets when coded alone, byte for byte.  This lets a batch of many files coded in one call single out
 * the files that need a fallback.  Out-of-range symbols (CZ_ERR_SYMBOL_RANGE) and NaN logits still fail the call.
 * RWKV-7 (floored alphabet) never has a zero-width token: it writes UINT64_MAX for every segment.  cap_segments < the call's
 * n_segments makes the call return CZ_ERR_INVALID.  NULL (the default when the model is created) restores failing with
 * CZ_ERR_ZERO_WIDTH; first_zw_out != NULL with cap_segments == 0 is CZ_ERR_INVALID. */
int cz_model_set_zero_width_out(cz_model *m, uint64_t *first_zw_out, size_t cap_segments);

/* Per-token code lengths.  With a sink set, cz_encode / cz_encode_dev write, for every global coded index i of the call:
 *   c_lo_out[i], c_hi_out[i]  the interval token i was coded with (c_lo == c_hi for a zero-width token, which only a call with the
 *                             zero-width sink set can return);  30 - log2(c_hi - c_lo) is its exact code length before coder overhead;
 *   entropy_out[i]            the expected code length of the distribution token i was coded from (cz_cdf_entropy), in the alphabet the
 *                             call codes with (cz_model_set_pdf_floor applies).
 * Any of the three may be NULL; all NULL (the default when the model is created) is off, and then the call launches exactly what it
 * launches without this function.  The sinks are written only when the call returns CZ_OK.  cap_tokens < the call's n_tokens makes the
 * call return CZ_ERR_INVALID; a non-NULL pointer with cap_tokens == 0 is CZ_ERR_INVALID.  Both architectures.  cz_decode, cz_xe_bits,
 * the session shim and cz_chunk_logits are unaffected. */
int cz_model_set_code_length_out(cz_model *m, uint32_t *c_lo_out, uint32_t *c_hi_out, double *entropy_out, size_t cap_tokens);

/* Preset dictionary.  With symbols D set (n > 0), cz_encode / cz_encode_dev / cz_decode code every segment g, coded tokens T_g, exactly
 * as they would code the token list D ++ T_g without a dictionary, except that the first n positions are not sent to the coder: the
 * intervals of T_g are, bit for bit, the last |T_g| intervals of a dictionary-less encode of D ++ T_g (BOS first, the reprime schedule
 * counted from the start of D, RWKV-7's literal escapes not stepping the model).  The stream must be decoded with the same dictionary.
 * SmolLM runs only the reprime chunk in which D ends and the chunks after it (at most one extra chunk of teacher-forced rows per
 * segment; that chunk's prime must fit max sequence length, else CZ_ERR_UNSUPPORTED); its decoder primes that chunk once for all
 * streams and copies the K/V rows.  RWKV-7 runs D once per call and copies the resulting state to every stream.
 * The symbols are copied and validated against the coded alphabet (CZ_ERR_SYMBOL_RANGE names the index).  NULL / 0 clears it (the
 * default when the model is created; every call then launches what it launches without this function).  A schedule with hint-prime
 * events is CZ_ERR_UNSUPPORTED while a dictionary is set.  cz_xe_bits, the session shim and cz_chunk_logits are unaffected; the
 * digest, code-length, zero-width sinks and the pdf floor work unchanged, indexed by global coded index. */
int cz_model_set_dictionary(cz_model *m, const uint32_t *symbols, size_t n);

/* Match model of order K (1..16; 0 is off, the default when the model is created).  It applies to the following cz_encode,
 * cz_encode_dev and cz_decode calls on both architectures.  With t[0..n) the coded symbols of one segment (RWKV-7 literal escapes
 * included; BOS and a dictionary are not: the history is the segment's own symbols), HB = 18 hash bits and NB = 16 length buckets:
 *   key(i), i >= K      h = 0x811C9DC5; for x in t[i-K .. i-1], oldest first: h = (h ^ x) * 0x01000193 mod 2^32;
 *                       key = (h * 0x9E3779B1 mod 2^32) >> (32 - HB)
 *   candidate           j(i) = max{ j : K <= j < i, key(j) == key(i) } in the same segment (a table of 2^HB positions per stream)
 *   length              len = the number of k = 0, 1, ... for which t[j-1-k] == t[i-1-k] (stopping at the first difference or at the
 *                       segment's start), at most K + NB - 1.  len < K (a hash collision) or no candidate: no prediction.  Otherwise
 *                       the prediction is pred = t[j], in bucket b = len - K
 *   weight              hits_b / tries_b = right / all predictions of bucket b at earlier positions of the segment;
 *                       p16 = clamp(((2 hits_b + 1) << 16) / (2 tries_b + 2), 1, 65535) (integer division), W = p16 << 14
 *   intervals of t[i]   with a prediction, first the flag: [0, W) if t[i] == pred (a hit), else [W, 2^30); then the model's interval
 *                       of t[i] unless it was a hit.
 * A hit's model interval is never coded, so the zero-width report (CZ_ERR_ZERO_WIDTH, cz_model_set_zero_width_out) names the first
 * non-hit token with an empty interval, by coded-token index.  cz_encode needs an output capacity of 8 bytes per token (4 without).
 * The code-length sink still reports the model's intervals.  A schedule with hint-prime events is CZ_ERR_UNSUPPORTED while the match
 * model is on.  cz_xe_bits, the session shim and cz_chunk_logits are unaffected; the digest, zero-width, code-length sinks, the pdf
 * floor and the dictionary work unchanged.  A stream must be decoded with the order it was encoded with (the container's MAT1 section).
 * Decode memory: 2^HB u32 positions per stream (1 MiB; 2 GiB at 2,048 streams), cleared at the start of each call.
 * order > 16 is CZ_ERR_INVALID. */
int cz_model_set_match(cz_model *m, uint32_t order);
/* Match-out sink: with the match model on, cz_encode / cz_encode_dev and cz_decode write, per global coded index i, the prediction
 * token i was coded with (pred_out[i], UINT32_MAX if none) and its flag weight W (w_out[i], 0 if none).  Encode and decode write the
 * same values.  Either pointer may be NULL; both NULL (the default) is off.  The sinks are written only when the call returns CZ_OK.
 * cap_tokens < the call's n_tokens makes the call return CZ_ERR_INVALID; a non-NULL pointer with cap_tokens == 0 is CZ_ERR_INVALID. */
int cz_model_set_match_out(cz_model *m, uint32_t *pred_out, uint32_t *w_out, size_t cap_tokens);

typedef struct {
  const uint32_t *prime;     /* tail(history, 511-|hint|) ++ hint, built by the caller or cz_xe_make_prime */
  uint32_t prime_len;
  const uint32_t *targets;
  uint32_t n_targets;
} cz_xe_job;
/* paired baseline / hint-conditioned streams of the agentic gate: all jobs run as one batch */
int cz_xe_bits(cz_model *m, const cz_xe_job *jobs, size_t n_jobs, double *bits_out);

/* teacher-forced logits of one chunk (prime ++ targets[:-1]) for tests: logits_out[n_targets][vocab] */
int cz_chunk_logits(cz_model *m, const uint32_t *prime, size_t prime_len, const uint32_t *targets, size_t n_targets,
                    float *logits_out);

/* ---------------------------------------------------------------- container (host-only) */
typedef struct {
  uint32_t bos_token_id;
  uint64_t token_count;
  uint64_t orig_len_bytes;
  uint8_t model_hash16[16];
  uint8_t tokenizer_hash16[16];
  uint8_t orig_hash16[16];
  uint32_t reserved_flags;
  uint32_t context_window;
  uint32_t vocab_size;
  uint32_t model_file_repr_len;
  uint32_t reprime_interval;
} cz_header_v2;

#define CZ_FLAG_AGENT_USED (1u << 0)
#define CZ_FLAG_AGENT_MOCK (1u << 1)
#define CZ_FLAG_AGENT_GATES (1u << 2)
#define CZ_FLAG_SEGMENTS (1u << 8) /* extension: a "SEG1" table follows the gates section (DESIGN.md) */
#define CZ_FLAG_STORED (1u << 9)   /* extension: the payload is the original bytes, uncoded.  Written by the file-level compress()
                                      when the SmolLM coder meets a symbol of mass < 2^-30 (CZ_ERR_ZERO_WIDTH: softmax_pdf has no
                                      floor, src/main.rs:2295; the reference would emit a corrupt stream there, SURVEY 7.3a) */
#define CZ_FLAG_PDF_FLOOR (1u << 10) /* extension: the payload was coded with the floored SmolLM pdf (CZ_CDF_SMOLLM_FLOOR,
                                        cz_model_set_pdf_floor).  Written by compress(on_zero_width="floor") when the unfloored pdf
                                        meets a zero-width symbol; never together with CZ_FLAG_STORED, never on RWKV-7 */
#define CZ_FLAG_DICTIONARY (1u << 11) /* extension: the payload was coded with a preset dictionary (cz_model_set_dictionary); a "DIC1"
                                         section names it, after the SEG1 table (or where it would be) and before the payloads.
                                         Never together with CZ_FLAG_STORED */
#define CZ_FLAG_MATCH (1u << 12) /* extension: the payload was coded with the match model (cz_model_set_match); a "MAT1" section gives
                                    its order, after the DIC1 section (or where it would be) and before the payloads.  Never together
                                    with CZ_FLAG_STORED */

size_t cz_container_header_size(const cz_header_v2 *h);
/* writes header (+repr); returns bytes written or 0 if cap is too small */
size_t cz_container_write_header(uint8_t *buf, size_t cap, const cz_header_v2 *h, const uint8_t *repr);
/* returns bytes consumed or 0 on parse error; *repr_off = offset of the repr string */
size_t cz_container_read_header(const uint8_t *buf, size_t len, cz_header_v2 *h, size_t *repr_off);
/* AGT2 gate records, one byte each: gate | cand<<1 | budget<<3 (src/main.rs:658-670) */
size_t cz_container_write_gates(uint8_t *buf, size_t cap, const uint8_t *records, size_t n);
/* accepts AGT2 and legacy AGTB (src/main.rs:2469-2484); returns bytes consumed, 0 on error */
size_t cz_container_read_gates(const uint8_t *buf, size_t len, uint8_t *records, size_t cap, size_t *n_records);
/* segment table: "SEG1" varint n_segments, varint engine, then per segment varint n_tokens, varint n_bytes */
size_t cz_container_write_segments(uint8_t *buf, size_t cap, int engine, const uint64_t *seg_tokens,
                                   const uint64_t *seg_bytes, size_t n);
size_t cz_container_read_segments(const uint8_t *buf, size_t len, int *engine, uint64_t *seg_tokens,
                                  uint64_t *seg_bytes, size_t cap, size_t *n);
/* dictionary section: "DIC1" varint n_symbols, then the BLAKE3-128 of the symbols as little-endian u32 (16 bytes) */
size_t cz_container_write_dictionary(uint8_t *buf, size_t cap, uint64_t n_symbols, const uint8_t hash16[16]);
size_t cz_container_read_dictionary(const uint8_t *buf, size_t len, uint64_t *n_symbols, uint8_t hash16[16]);
/* match-model section: "MAT1" varint order.  The reader returns 0 for a truncated section or an order outside [1, 16] */
size_t cz_container_write_match(uint8_t *buf, size_t cap, uint32_t order);
size_t cz_container_read_match(const uint8_t *buf, size_t len, uint32_t *order);
uint32_t cz_flags_pack(int agent_used, int agent_mock, int gates_present, uint32_t agent_chunk);
/* BLAKE3-128 of a buffer (src/main.rs:901-920 use blake3 truncated to 16 bytes) */
void cz_blake3_16(const uint8_t *data, size_t len, uint8_t out16[16]);

/* ---------------------------------------------------------------- host schedule (for tests / INTEGRATION) */
/* Expands the reference's loop (src/main.rs:1979, 2275-2290) into independent chunks.
 * For segment-relative coded index i in [0,n): chunk boundaries and prime windows.  Returns the number
 * of chunks; fills up to cap entries of: first coded index, number coded, prime start (index into the
 * segment's token list incl. BOS at 0), prime length. */
size_t cz_schedule_chunks(uint64_t n_tokens, uint32_t context, uint32_t reprime_interval, uint64_t *first,
                          uint32_t *n_coded, uint64_t *prime_start, uint32_t *prime_len, size_t cap);
/* The same under a dictionary of n_prefix symbols (cz_model_set_dictionary): the chunks of cz_schedule_chunks(n_prefix + n_tokens)
 * that code at least one of the n_tokens, first counted from the first of them, and the prefix positions of the chunk in which the
 * dictionary ends added to its prime.  prime_start indexes the list BOS ++ dictionary ++ tokens. */
size_t cz_schedule_chunks_prefixed(uint64_t n_tokens, uint64_t n_prefix, uint32_t context, uint32_t reprime_interval, uint64_t *first,
                                   uint32_t *n_coded, uint64_t *prime_start, uint32_t *prime_len, size_t cap);

/* ---------------------------------------------------------------- test hooks (not part of the drop-in surface) */
/* one dense contraction C[M,N] (+)= A[M,K] B[N,K]^T through the chosen engine on host buffers; epi: 0 store f32,
 * 1 add f32, 2 swiglu->bf16 (B rows packed bn/2 gate + bn/2 up), 3 store bf16; bn: 192 or 256 */
int cz_test_gemm(cz_ctx *ctx, int engine, int M, int N, int K, const uint16_t *a_bf16, const uint16_t *b_bf16, int epi,
                 int bn, void *c_inout, int ldc);

/* the fused residual-add + RMSNorm pair (tcgen05 engine, N a multiple of 192): x[M,N] += A[M,K] B[N,K]^T with
 * xb = bf16(x * w_next) and per-row partial sums of squares (producer epilogue), then out[M,N2] = bf16(rowscale * (xb B2[N2,N]^T))
 * with rowscale = 1 / sqrt(sum(x^2) / N + eps) (consumer epilogue).  Outputs: x (in place), xb_out [M][N], ssq_out [M][(N/192)*3],
 * out2 [M][N2] (bf16). */
int cz_test_gemm_norm(cz_ctx *ctx, int M, int N, int K, int N2, const uint16_t *a_bf16, const uint16_t *b_bf16, const uint16_t *b2_bf16,
                      const float *w_next, float eps, float *x_inout, uint16_t *xb_out, float *ssq_out, uint16_t *out2);

/* one causal GQA attention pass of the tcgen05 kernel over one sequence (q [n_pos][nh*64], k / v [n_pos][nkv*64], bf16, RoPE already
 * applied): mode 0 = teacher-forced 128-position tiles, mode 1 = every position as a single-row decode tile; out [n_pos][nh*64] bf16 */
int cz_test_attention(cz_ctx *ctx, int n_pos, int nh, int nkv, const uint16_t *q_bf16, const uint16_t *k_bf16,
                      const uint16_t *v_bf16, int mode, uint16_t *out_bf16);

/* one WKV-7 scan (csrc/rwkv7.cu wkv7_scan_kernel<layer0>) over R rows of width C = 64 H (H <= 16): stream s walks rows
 * row_begin[s] .. row_end[s]-1 in order from state slot stream_slot[s]; stream_active (nullable) skips streams whose flag is 0.
 * rows [7][R][C] = r, k, v, w-LoRA, a-LoRA, v-LoRA, g (f32); vecs [8][C] = w0, a0, v0, k_k, k_a, r_k, gn_w, gn_b; v_first [R][C] in/out
 * (written with layer0, read without); state [n_slots][H][4096] in/out in the kernel's layout (row i, column j of a head's 64x64
 * matrix at (j/4)*256 + i*4 + j%4); out_bf16 [R][C] in/out (rows no active stream covers keep their contents) */
int cz_test_wkv7_scan(cz_ctx *ctx, int layer0, int R, int H, int n_streams, const int *row_begin, const int *row_end, const int *stream_slot,
                      const int *stream_active, int n_slots, const float *rows, float *v_first, const float *vecs, float *state,
                      uint16_t *out_bf16);
/* one LayerNorm + token-shift mix (rwkv_ln_mix, nmix 1 or 6) over R rows of width C <= 1024: x [R][C], lnw / lnb [C], mu [nmix][C],
 * per row prev_row (-1: the previous token is state_in[slot]), slot and flags (bit 0 writes state_out[slot], bit 1 suppresses it);
 * state_in [n_slots][C]; state_out [n_slots][C] in/out, or with in_place the kernel reads and writes one buffer that starts as
 * state_in.  form 0 runs what the model would run, 1 forces the element-per-lane kernel; *form_used = elements per lane of the kernel
 * that ran (1 or 8).  out_bf16 [nmix][R][C]. */
int cz_test_rwkv_ln_mix(cz_ctx *ctx, int nmix, int form, int in_place, int R, int C, int n_slots, const float *x, const float *lnw,
                        const float *lnb, const float *mu, const int *prev_row, const int *slot, const int *flags, const float *state_in,
                        float *state_out, float eps, uint16_t *out_bf16, int *form_used);

/* the CDF kernels' fast paths against the originals (csrc/cdf_fast.cuh): (1) every non-negative f32 argument pattern of
 * expf(-(max - logit)): the integer-conversion path must give the bits of the conversion path wherever it is taken; `checksum` =
 * sum over the patterns b of bits(expf(-float(b))) * (2 b + 1) mod 2^64 (NaN results as 0x7fc00000), which the CPU oracle reproduces
 * with its glibc-verified expf (czo_expf_checksum); (2) the reciprocal-based division against the IEEE division on random operands */
int cz_test_expf_exhaustive(cz_ctx *ctx, uint64_t *mismatches, uint64_t *checksum, uint64_t *first_bad);
int cz_test_div_random(cz_ctx *ctx, uint64_t seed, uint64_t n_pairs, uint64_t *mismatches);
/* what the last encode-side CDF batch (cz_cdf_bounds or the executor) did with the e-cache -- the compact copy of e_v, v <= coded
 * symbol, that the stats pass leaves for the prefix walk (csrc/cdf_kernels.cu): *state = 1 the prefix walk read the cache, 0 the batch
 * did not fit its capacity and the walk read the logits, -1 no cache was set up for that batch; *groups = 64-byte groups used */
int cz_test_cdf_ecache_state(cz_ctx *ctx, int *state, uint64_t *groups);

#ifdef __cplusplus
}
#endif
#endif /* CANDLEZIP_B200_H */
