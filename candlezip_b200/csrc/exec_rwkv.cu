// RWKV-7 schedule executor: batched encode, lock-step batched decode, paired XE scan and the batch-of-1 session shim.
//
// Replaces the RWKV legs of the reference's loops: encode src/main.rs:1979, 2301-2326, 2344-2350; decode 2706-2864;
// gate cross-entropy 1753-1787; Rwkv7Session src/models.rs:151-179.  Differences from the SmolLM executor (exec.cu):
//   * no context re-prime (the `if backend=="smollm"` guard at main.rs:2275): a stream's state runs over its whole segment, so
//     the unit of work is a UNIT = (stepped token list, coded columns); a gated hint prime resets the state
//     (models.rs:162-170) and therefore simply starts a new unit;
//   * the coded alphabet is V + 256 literal-escape symbols; a literal symbol does not step the model (main.rs:2347-2349,
//     2832-2834), so several coded columns can share one logits row;
//   * time is processed in SLABS of T steps of every live unit (rwkv7.cu), the recurrent state living in HBM between slabs.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "cdf_fast.cuh"
#include "coder.cuh"
#include "match.h"
#include "model.h"

namespace cz {
int launch_cdf_cols(cz_ctx *ctx, int op, int mode, const float *logits_dev, size_t V, size_t M, size_t ld,
                    const uint32_t *arg_dev, uint32_t *sym_out_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev,
                    double *xe_dev, cudaStream_t stream, const int *colmax_dev = nullptr);
int launch_cdf_entropy(cz_ctx *ctx, int mode, const float *logits_dev, size_t V, size_t M, size_t ld, double *h_dev, cudaStream_t stream);
int fetch_device_status(cz_ctx *ctx, unsigned long long *err_index_dev, unsigned long long *err_index_out);
int launch_decode_step(cz_ctx *ctx, int mode, const float *logits, int V, size_t ld, int n_lanes, const uint8_t *payload,
                       const uint64_t *seg_off, const uint64_t *seg_start, uint64_t coded_index, void *decoder_state, uint32_t *ids_out,
                       uint32_t *next_tok, const int *colmax, cudaStream_t st, const unsigned long long *ctr, const MatchDecView *mv);
int launch_decoder_init(cz_ctx *ctx, const uint8_t *payload, const uint64_t *seg_off, int n_lanes, void *decoder_state, cudaStream_t st);
size_t decoder_state_bytes();
int launch_set_ctr(cz_ctx *ctx, unsigned long long *ctr, unsigned long long a, unsigned long long b, cudaStream_t st);
int launch_advance_ctr(cz_ctx *ctx, unsigned long long *ctr, cudaStream_t st);
}  // namespace cz

namespace czk {

// tok[r] = src[r] >= 0 ? ids[src[r]] : (src[r] == -1 ? bos : extra[-2 - src[r]])
__global__ void rw_gather_tokens_kernel(const long long *__restrict__ src, const uint32_t *__restrict__ ids,
                                        const uint32_t *__restrict__ extra, uint32_t bos, uint32_t *__restrict__ tok, int n) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  long long s = src[r];
  tok[r] = s >= 0 ? ids[s] : (s == -1 ? bos : extra[-2 - s]);
}
__global__ void rw_gather_syms_kernel(const uint32_t *__restrict__ col_sym, const unsigned long long *__restrict__ idx,
                                      uint32_t *__restrict__ out, int n) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) out[c] = col_sym[idx[c]];
}
__global__ void rw_scatter_bounds_kernel(const uint32_t *__restrict__ lo, const uint32_t *__restrict__ hi,
                                         const unsigned long long *__restrict__ idx, uint32_t *__restrict__ lo_out,
                                         uint32_t *__restrict__ hi_out, int n) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  lo_out[idx[c]] = lo[c];
  hi_out[idx[c]] = hi[c];
}
__global__ void rw_scatter_xe_kernel(const double *__restrict__ xe, const unsigned long long *__restrict__ idx, double *__restrict__ out, int n) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n) out[idx[c]] = xe[c];
}
__global__ void rw_sum_bits_kernel(const double *__restrict__ bits, const uint64_t *__restrict__ job_off, double *__restrict__ out, int n_jobs) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_jobs) return;
  double acc = 0.0;  // sequential f64, like `bits += ...` in src/main.rs:1781
  for (uint64_t t = job_off[j]; t < job_off[j + 1]; t++) acc = __dadd_rn(acc, bits[t]);
  out[j] = acc;
}
// stepwise decode: which streams step the model after this symbol (main.rs:2832-2834), and with which token
__global__ void rw_decode_flags_kernel(const uint32_t *__restrict__ sym, uint32_t V, const uint64_t *__restrict__ seg_start,
                                       const unsigned long long *__restrict__ ctr, int n_lanes, int *__restrict__ flags,
                                       int *__restrict__ active, uint32_t *__restrict__ tok) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_lanes) return;
  const uint64_t coded_index = ctr[0];
  const uint64_t len = seg_start[s + 1] - seg_start[s];
  const bool act = coded_index + 1 < len && sym[s] < V;  // the step after a stream's last symbol is never needed
  active[s] = act ? 1 : 0;
  flags[s] = act ? 1 : 3;
  tok[s] = act ? sym[s] : 0u;
}
// copy the freshly computed logits columns (and column maxima) of the streams that stepped into the persistent buffer
__global__ void rw_commit_logits_kernel(const float *__restrict__ fresh, float *__restrict__ keep, size_t ld, size_t total,
                                        const int *__restrict__ active, const int *__restrict__ cm_fresh, int *__restrict__ cm_keep,
                                        int n_lanes) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (size_t)n_lanes && active[i] && cm_fresh) cm_keep[i] = cm_fresh[i];
  if (i >= total) return;
  const size_t col = i % ld;
  if (col < (size_t)n_lanes && active[col]) keep[i] = fresh[i];
}

// Preset dictionary: copies the recurrent state of slot 0 -- the WKV state [L][cap][H * 4096] and the token-shift rows xa / xf
// [L][cap][C] of the current ping-pong side -- to slots [1, n), so every stream starts from the state the dictionary left.
// 16-byte pieces; blockIdx.y = 0: WKV state, 1: xa, 2: xf.
__global__ void rwkv_state_broadcast_kernel(float *__restrict__ S, float *__restrict__ xa, float *__restrict__ xf, int L, size_t cap,
                                            size_t s4, size_t c4, int n) {
  const size_t per = (size_t)(n - 1);
  const size_t w4 = blockIdx.y == 0 ? s4 : c4;  // 16-byte pieces per slot and layer
  float4 *base = (float4 *)(blockIdx.y == 0 ? S : blockIdx.y == 1 ? xa : xf);
  const size_t total = (size_t)L * per * w4;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t e = i % w4, r = i / w4, g = 1 + r % per, l = r / per;
    float4 *layer = base + l * cap * w4;
    layer[g * w4 + e] = layer[e];
  }
}

}  // namespace czk

namespace cz {

struct RwUnit {
  std::vector<long long> step_src;  // token source of every model step (gather encoding)
  std::vector<uint32_t> col_step;   // per coded column: index of the step whose logits code it (non-decreasing)
  uint64_t col0 = 0;                // global id of the unit's first column
};

// appends the stepped tokens / columns of a run of coded tokens tok[0..n) (host copy) whose global column ids start at col0.
// `first_src`: sources of the tokens stepped before the first coded token (BOS, or a hint prime).  src_of(j) = gather code of tok j.
template <class F>
static void build_unit(RwUnit &u, const std::vector<long long> &first_src, const uint32_t *tok, size_t n, uint32_t V, uint64_t col0, F src_of) {
  u.step_src = first_src;
  u.col_step.resize(n);
  u.col0 = col0;
  for (size_t j = 0; j < n; j++) {
    u.col_step[j] = (uint32_t)(u.step_src.size() - 1);
    if (j + 1 < n && tok[j] < V) u.step_src.push_back(src_of(j));  // literals do not step; the last token's step is never used
  }
}

// rows of one slab when the schedule sets no max_batch_tokens (encode), and the bound on a decode prime slab
static const size_t kSlabRows = 262144;

// Preset dictionary (cz_model_set_dictionary): a stream of D ++ T steps BOS and the in-vocabulary symbols of D before it codes T[0]
// (literal escapes never step the model).  Every stream of a call shares that history, so it runs ONCE: `feed` = BOS and all but the
// last in-vocabulary symbol, run for one slot; each stream then steps `last` itself (the gather code of that symbol in the dictionary,
// which is the `extra` buffer, or -1 = BOS when D has no in-vocabulary symbol, in which case `feed` is empty).
struct RwPrefix {
  std::vector<uint32_t> feed;
  long long last = -1;
};
static RwPrefix rwkv_prefix(const cz_model *m, uint32_t bos) {
  RwPrefix p;
  const std::vector<uint32_t> &d = m->dictionary;
  for (size_t k = 0; k < d.size(); k++)
    if (d[k] < (uint32_t)m->cfg.vocab) {
      p.feed.push_back(p.last == -1 ? bos : d[(size_t)(-2 - p.last)]);  // (a gather code is negative: -1 is BOS, -2 - k is d[k])
      p.last = -2 - (long long)k;
    }
  return p;
}

// runs p.feed through slot 0 of the freshly reset `stt` in slabs of at most max_rows rows, then copies slot 0's state to slots [1, n)
static int rwkv_prefix_state(cz_model *m, RwkvState &stt, const RwPrefix &p, size_t n, size_t max_rows, cudaStream_t st) {
  if (p.feed.empty()) return CZ_OK;  // the zero state
  cz_ctx *ctx = m->ctx;
  const cz_model_config &c = m->cfg;
  Workspace &ws = m->ws;
  RwkvWs &rw = m->rws;
  const int zero = 0;
  for (size_t k0 = 0; k0 < p.feed.size(); k0 += max_rows) {
    const size_t T = std::min(max_rows, p.feed.size() - k0);
    CZ_TRY(ensure_workspace(m, T, 1, 0));
    CZ_TRY(rwkv_ensure_ws(m, T, 1));
    std::vector<int> prev(T), slot(T, 0), flags(T, 0);
    for (size_t k = 0; k < T; k++) prev[k] = (int)k - 1;
    flags[T - 1] = 1;
    const int re = (int)T;
    CZ_CUDA_TRY(cudaMemcpyAsync(ws.tok, p.feed.data() + k0, T * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.prev_row, prev.data(), T * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.slot, slot.data(), T * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.flags, flags.data(), T * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_begin, &zero, 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_end, &re, 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.stream_slot, &zero, 4, cudaMemcpyHostToDevice, st));
    CZ_TRY(rwkv_forward(m, (int)T, 1, stt, /*in_place=*/false, nullptr, st));
    CZ_CUDA_TRY(cudaStreamSynchronize(st));  // the staging vectors are stack-owned
  }
  if (n > 1) {
    const size_t C = c.d_model, H = C / 64;
    CZ_LAUNCH(ctx, CZ_K_OTHER,
              (czk::rwkv_state_broadcast_kernel<<<dim3(592, 3), 256, 0, st>>>(stt.S, stt.xa[stt.cur], stt.xf[stt.cur], c.n_layers, stt.cap,
                                                                             H * 4096 / 4, C / 4, (int)n)));
    CZ_CHECK_LAUNCH();
  }
  return CZ_OK;
}

// The units of one stream of n coded tokens under the schedule's hint-prime events (n_segments == 1 when there are any): unit u
// covers coded indices [begin, next unit's begin) and starts from a zero state primed with BOS (event -1) or with the prime of
// `event`.  Of several events at one index the last wins; an event at an index already passed (out of order) is skipped and one at
// i >= n never applies.  The encoder and the decoder both plan with this, so they apply the same event at the same index.
struct RwCut {
  uint64_t begin;
  int event;
};
static int rwkv_plan_units(const cz_schedule *s, uint64_t n, uint32_t V, std::vector<RwCut> &cuts) {
  cuts.clear();
  uint32_t ev = 0;
  for (uint64_t cur = 0; cur < n;) {
    int at = -1;
    for (; ev < s->n_events && s->events[ev].i <= cur; ev++) {
      const cz_prime_event &e = s->events[ev];
      if (e.i != cur) continue;
      bool any = e.hist_take > 0;  // a history tail is never empty: BOS pads it
      for (uint32_t k = 0; k < e.prime_len && !any; k++) any = e.prime[k] < V;
      if (!any) {
        set_error("rwkv: hint prime has no in-vocabulary token");
        return CZ_ERR_INVALID;
      }
      at = (int)ev;
    }
    cuts.push_back({cur, at});
    cur = ev < s->n_events && s->events[ev].i < n ? s->events[ev].i : n;
  }
  return CZ_OK;
}

// Gather codes (rw_gather_tokens_kernel) of the prime of hint event e applied at coded index cur of a stream that starts at a: the
// last hist_take symbols below V among ids[a, cur) in order, preceded by BOS when there are fewer (S[0] = BOS), then the event's
// explicit tokens below V, which the caller holds at extra[ev_off ..).  Literal escapes are filtered out (main.rs:2139-2141).
// ids: the host's copy of at least ids[a, cur).
static void rwkv_event_prime(const cz_prime_event &e, const uint32_t *ids, uint64_t a, uint64_t cur, uint32_t V, size_t ev_off,
                             std::vector<long long> &first) {
  first.clear();
  for (uint64_t t = cur; t > a && first.size() < e.hist_take; t--)
    if (ids[t - 1] < V) first.push_back((long long)(t - 1));
  if (first.size() < e.hist_take) first.push_back(-1ll);
  std::reverse(first.begin(), first.end());
  for (uint32_t k = 0; k < e.prime_len; k++)
    if (e.prime[k] < V) first.push_back(-2 - (long long)(ev_off + k));
}

struct RwOut {
  int op = czk::OP_BOUNDS;
  const uint32_t *col_sym = nullptr;  // device, indexed by global column id
  uint32_t *lo = nullptr, *hi = nullptr;
  double *xe = nullptr;
  double *ent = nullptr;         // OP_BOUNDS: also each column's coding-distribution entropy (cdf_entropy_kernel), by global column id
  float *logits_host = nullptr;  // test hook: [n_cols][V] row-major on the host (single unit)
  bool digest = false;           // f-4: hash every column's logits into the model's digest buffer at its global coded index
};

// prefix (nullable): the units start from the state it leaves (rwkv_prefix_state) instead of the zero state
static int rwkv_run_units(cz_model *m, std::vector<RwUnit> &units, const uint32_t *ids_dev, const uint32_t *extra_dev, uint32_t bos,
                          const RwOut &o, size_t max_rows, cudaStream_t st, const RwPrefix *prefix = nullptr) {
  cz_ctx *ctx = m->ctx;
  const cz_model_config &c = m->cfg;
  const size_t U = units.size(), V = c.vocab;
  if (U == 0) return CZ_OK;
  size_t max_steps = 0;
  for (auto &u : units) max_steps = std::max(max_steps, u.step_src.size());
  if (max_rows == 0) max_rows = kSlabRows;
  const size_t Tw = std::max<size_t>(1, std::min(max_steps, max_rows / U));
  CZ_TRY(rwkv_state_reset(m, m->rstate, U, st));
  if (prefix) CZ_TRY(rwkv_prefix_state(m, m->rstate, *prefix, U, max_rows, st));
  std::vector<long long> src;
  std::vector<int> prev_row, slot, flags, row_begin, row_end, sslot, logit_rows;
  std::vector<unsigned long long> out_idx;
  std::vector<size_t> col_ptr(U, 0);
  GrowBuf &d_src = m->sb[SB_SRC], &d_oidx = m->sb[SB_RW_OIDX], &d_syms = m->sb[SB_RW_SYMS], &d_lo = m->sb[SB_RW_LO], &d_hi = m->sb[SB_RW_HI],
          &d_xe = m->sb[SB_RW_XE];
  for (size_t t0 = 0; t0 < max_steps; t0 += Tw) {
    src.clear(); prev_row.clear(); slot.clear(); flags.clear(); row_begin.clear(); row_end.clear(); sslot.clear();
    logit_rows.clear(); out_idx.clear();
    for (size_t ui = 0; ui < U; ui++) {
      RwUnit &u = units[ui];
      if (u.step_src.size() <= t0) continue;
      const size_t t1 = std::min(u.step_src.size(), t0 + Tw);
      const int rb = (int)src.size();
      for (size_t t = t0; t < t1; t++) {
        src.push_back(u.step_src[t]);
        prev_row.push_back(t == t0 ? -1 : (int)src.size() - 2);
        slot.push_back((int)ui);
        flags.push_back(t + 1 == t1 ? 1 : 0);
      }
      row_begin.push_back(rb);
      row_end.push_back((int)src.size());
      sslot.push_back((int)ui);
      size_t &cp = col_ptr[ui];
      while (cp < u.col_step.size() && u.col_step[cp] < t1) {
        logit_rows.push_back(rb + (int)(u.col_step[cp] - t0));
        out_idx.push_back(u.col0 + cp);
        cp++;
      }
    }
    const size_t R = src.size(), NS = sslot.size(), NL = logit_rows.size();
    if (R == 0) break;
    CZ_TRY(ensure_workspace(m, R, NL, 0));
    CZ_TRY(rwkv_ensure_ws(m, R, NS));
    CZ_TRY(d_src.reserve(R * 8, st));
    CZ_TRY(d_oidx.reserve(NL * 8 + 16, st));
    Workspace &ws = m->ws;
    RwkvWs &rw = m->rws;
    // ---- upload the slab's metadata through the pinned staging buffer ----
    if (!ws.stage_ev) CZ_CUDA_TRY(cudaEventCreateWithFlags(&ws.stage_ev, cudaEventDisableTiming));
    else CZ_CUDA_TRY(cudaEventSynchronize(ws.stage_ev));
    const size_t bytes = R * 20 + NS * 12 + NL * 12 + 256;
    CZ_TRY(ensure_stage(m, bytes));
    char *h = (char *)ws.h_stage;
    size_t off = 0;
    auto put = [&](void *dst_dev, const void *host, size_t nbytes) -> int {
      if (nbytes == 0) return CZ_OK;
      memcpy(h + off, host, nbytes);
      CZ_CUDA_TRY(cudaMemcpyAsync(dst_dev, h + off, nbytes, cudaMemcpyHostToDevice, st));
      off += (nbytes + 15) & ~(size_t)15;
      return CZ_OK;
    };
    CZ_TRY(put(d_src.p, src.data(), R * 8));
    CZ_TRY(put(rw.prev_row, prev_row.data(), R * 4));
    CZ_TRY(put(rw.slot, slot.data(), R * 4));
    CZ_TRY(put(rw.flags, flags.data(), R * 4));
    CZ_TRY(put(rw.row_begin, row_begin.data(), NS * 4));
    CZ_TRY(put(rw.row_end, row_end.data(), NS * 4));
    CZ_TRY(put(rw.stream_slot, sslot.data(), NS * 4));
    CZ_TRY(put(ws.logit_rows, logit_rows.data(), NL * 4));
    CZ_TRY(put(d_oidx.p, out_idx.data(), NL * 8));
    CZ_CUDA_TRY(cudaEventRecord(ws.stage_ev, st));
    CZ_LAUNCH(ctx, CZ_K_OTHER,
              (czk::rw_gather_tokens_kernel<<<(unsigned)ceil_div(R, 256), 256, 0, st>>>(d_src.as<long long>(), ids_dev, extra_dev, bos, ws.tok, (int)R)));
    CZ_CHECK_LAUNCH();
    CZ_TRY(rwkv_forward(m, (int)R, (int)NS, m->rstate, /*in_place=*/false, nullptr, st));
    if (NL == 0) continue;
    CZ_TRY(rwkv_final_norm_gather(m, (int)NL, st));
    if (o.logits_host) {  // test hook: dump the logits of every column
      CZ_TRY(ensure_logits(m, 256));
      const size_t ld_c = 256;
      std::vector<float> tmp(V * ld_c);
      for (size_t c0 = 0; c0 < NL; c0 += ld_c) {
        const size_t nc = std::min(ld_c, NL - c0);
        CZ_TRY(lm_head(m, (int)c0, (int)nc, ws.logits[0], ld_c, st));
        CZ_CUDA_TRY(cudaMemcpyAsync(tmp.data(), ws.logits[0], V * ld_c * 4, cudaMemcpyDeviceToHost, st));
        CZ_CUDA_TRY(cudaStreamSynchronize(st));
        for (size_t j = 0; j < nc; j++) {
          float *dst = o.logits_host + (size_t)(out_idx[c0 + j] - units[0].col0) * V;
          for (size_t v = 0; v < V; v++) dst[v] = tmp[v * ld_c + j];
        }
      }
      continue;
    }
    CZ_TRY(ensure_logits(m, NL));
    CZ_TRY(d_syms.reserve(NL * 4 + 16, st));
    CZ_TRY(d_lo.reserve(NL * 4 + 16, st));
    CZ_TRY(d_hi.reserve(NL * 4 + 16, st));
    CZ_TRY(d_xe.reserve(NL * 8 + 16, st));
    CZ_LAUNCH(ctx, CZ_K_OTHER,
              (czk::rw_gather_syms_kernel<<<(unsigned)ceil_div(NL, 256), 256, 0, st>>>(o.col_sym, d_oidx.as<unsigned long long>(),
                                                                                      d_syms.as<uint32_t>(), (int)NL)));
    CZ_CHECK_LAUNCH();
    for (size_t c0 = 0; c0 < NL; c0 += ws.ld_sub) {
      const size_t nc = std::min(ws.ld_sub, NL - c0);
      bool have_max = false;
      CZ_TRY(lm_head(m, (int)c0, (int)nc, ws.logits[0], ws.ld_sub, st, ws.colmax, &have_max));
      if (o.digest)  // (before the CDF pass, which caches expf values in the logits' slots)
        CZ_TRY(launch_logits_digest(ctx, ws.logits[0], V, nc, ws.ld_sub, m->sb[SB_CV].p, m->sb[SB_DIGEST].as<uint8_t>(), 0,
                                    d_oidx.as<unsigned long long>() + c0, nullptr, nullptr, st));
      CZ_TRY(launch_cdf_cols(ctx, o.op, CZ_CDF_RWKV_LITERALS, ws.logits[0], V, nc, ws.ld_sub, d_syms.as<uint32_t>() + c0, nullptr,
                             d_lo.as<uint32_t>() + c0, d_hi.as<uint32_t>() + c0, d_xe.as<double>() + c0, st,
                             have_max ? ws.colmax : nullptr));
      if (o.ent)  // (the per-column results of the encode pass are unused there: d_xe holds the entropies until the scatter)
        CZ_TRY(launch_cdf_entropy(ctx, CZ_CDF_RWKV_LITERALS, ws.logits[0], V, nc, ws.ld_sub, d_xe.as<double>() + c0, st));
    }
    if (o.op == czk::OP_XE || o.ent)
      CZ_LAUNCH(ctx, CZ_K_OTHER,
                (czk::rw_scatter_xe_kernel<<<(unsigned)ceil_div(NL, 256), 256, 0, st>>>(d_xe.as<double>(), d_oidx.as<unsigned long long>(),
                                                                                       o.op == czk::OP_XE ? o.xe : o.ent, (int)NL)));
    if (o.op != czk::OP_XE)
      CZ_LAUNCH(ctx, CZ_K_OTHER,
                (czk::rw_scatter_bounds_kernel<<<(unsigned)ceil_div(NL, 256), 256, 0, st>>>(d_lo.as<uint32_t>(), d_hi.as<uint32_t>(),
                                                                                           d_oidx.as<unsigned long long>(), o.lo, o.hi, (int)NL)));
    CZ_CHECK_LAUNCH();
  }
  return CZ_OK;
}

// ---- encode: fills lo/hi for every coded token (device arrays indexed by global coded index) -------------------------------
int rwkv_encode_bounds(cz_model *m, const uint32_t *ids_dev, const uint32_t *ids_host, size_t n_tokens, const cz_schedule *sched,
                       const uint32_t *extra_dev, const std::vector<size_t> &ev_off, uint32_t *lo_dev, uint32_t *hi_dev, double *ent_dev,
                       cudaStream_t st) {
  const uint32_t V = (uint32_t)m->cfg.vocab;
  std::vector<uint32_t> host_copy;
  if (!ids_host) {  // device-resident entry point: the host needs the ids to see which symbols are literal escapes
    host_copy.resize(n_tokens);
    CZ_CUDA_TRY(cudaMemcpyAsync(host_copy.data(), ids_dev, n_tokens * 4, cudaMemcpyDeviceToHost, st));
    CZ_CUDA_TRY(cudaStreamSynchronize(st));
    ids_host = host_copy.data();
  }
  std::vector<RwUnit> units;
  std::vector<RwCut> cuts;
  std::vector<long long> first;
  const RwPrefix prefix = rwkv_prefix(m, sched->bos);  // (a dictionary excludes events: extra_dev then holds the dictionary)
  for (uint32_t g = 0; g < sched->n_segments; g++) {
    const uint64_t a = sched->seg_start[g], b = sched->seg_start[g + 1];
    CZ_TRY(rwkv_plan_units(sched, b - a, V, cuts));
    for (size_t u = 0; u < cuts.size(); u++) {
      const uint64_t cur = a + cuts[u].begin, end = u + 1 < cuts.size() ? a + cuts[u + 1].begin : b;
      // BOS (main.rs:1916), or a gated hint prime, which restarts the state (main.rs:2137-2149 -> models.rs:162-170)
      if (cuts[u].event < 0) first.assign(1, prefix.last);
      else rwkv_event_prime(sched->events[cuts[u].event], ids_host, a, cur, V, ev_off[cuts[u].event], first);
      units.emplace_back();
      build_unit(units.back(), first, ids_host + cur, (size_t)(end - cur), V, cur, [&](size_t j) { return (long long)(cur + j); });
    }
  }
  RwOut o;
  o.op = czk::OP_BOUNDS;
  o.col_sym = ids_dev;
  o.lo = lo_dev;
  o.hi = hi_dev;
  o.ent = ent_dev;
  o.digest = m->digest_host != nullptr;  // (encode_core reserved the buffers: digest_begin)
  return rwkv_run_units(m, units, ids_dev, extra_dev, sched->bos, o, sched->max_batch_tokens, st, &prefix);
}

// ---- paired XE scan (main.rs:1753-1787) ---------------------------------------------------------------------------------------
int rwkv_xe_bits(cz_model *m, const cz_xe_job *jobs, size_t n_jobs, double *bits_out) {
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  const uint32_t V = (uint32_t)m->cfg.vocab;
  std::vector<uint32_t> extra, tgt;
  std::vector<uint64_t> job_off(n_jobs + 1, 0);
  std::vector<RwUnit> units;
  for (size_t j = 0; j < n_jobs; j++) {
    job_off[j + 1] = job_off[j] + jobs[j].n_targets;
    if (jobs[j].n_targets == 0) continue;
    std::vector<long long> first;
    for (uint32_t k = 0; k < jobs[j].prime_len; k++)
      if (jobs[j].prime[k] < V) {  // literals are filtered out of the prime (main.rs:1763-1765)
        first.push_back(-2 - (long long)extra.size());
        extra.push_back(jobs[j].prime[k]);
      }
    if (first.empty()) {
      set_error("xe job with targets needs a non-empty prime (the reference bails on an empty reprime)");
      return CZ_ERR_INVALID;
    }
    const size_t t0 = extra.size();
    extra.insert(extra.end(), jobs[j].targets, jobs[j].targets + jobs[j].n_targets);
    tgt.insert(tgt.end(), jobs[j].targets, jobs[j].targets + jobs[j].n_targets);
    units.emplace_back();
    build_unit(units.back(), first, jobs[j].targets, jobs[j].n_targets, V, job_off[j], [&](size_t q) { return -2 - (long long)(t0 + q); });
  }
  const size_t n_cols = tgt.size();
  GrowBuf &d_extra = m->sb[SB_EXTRA], &d_tgt = m->sb[SB_TGT], &d_bits = m->sb[SB_BITS], &d_joff = m->sb[SB_JOFF], &d_out = m->sb[SB_XOUT];
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  CZ_TRY(d_tgt.reserve(n_cols * 4 + 16, st));
  CZ_TRY(d_bits.reserve(n_cols * 8 + 16, st));
  CZ_TRY(d_joff.reserve((n_jobs + 1) * 8, st));
  CZ_TRY(d_out.reserve(n_jobs * 8, st));
  if (!extra.empty()) CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));
  if (n_cols) CZ_CUDA_TRY(cudaMemcpyAsync(d_tgt.p, tgt.data(), n_cols * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_joff.p, job_off.data(), (n_jobs + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));  // extra / tgt are stack-owned
  RwOut o;
  o.op = czk::OP_XE;
  o.col_sym = d_tgt.as<uint32_t>();
  o.xe = d_bits.as<double>();
  CZ_TRY(rwkv_run_units(m, units, nullptr, d_extra.as<uint32_t>(), 0, o, 0, st));
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::rw_sum_bits_kernel<<<(unsigned)ceil_div(n_jobs, 128), 128, 0, st>>>(d_bits.as<double>(), d_joff.as<uint64_t>(),
                                                                                     d_out.as<double>(), (int)n_jobs)));
  CZ_CHECK_LAUNCH();
  CZ_CUDA_TRY(cudaMemcpyAsync(bits_out, d_out.p, n_jobs * 8, cudaMemcpyDeviceToHost, st));
  return fetch_device_status(ctx, nullptr, nullptr);
}

// ---- test hook: logits of one unit --------------------------------------------------------------------------------------------
int rwkv_chunk_logits(cz_model *m, const uint32_t *prime, size_t prime_len, const uint32_t *targets, size_t n_targets, float *logits_out) {
  cudaStream_t st = m->ctx->stream;
  const uint32_t V = (uint32_t)m->cfg.vocab;
  std::vector<uint32_t> extra(prime, prime + prime_len);
  extra.insert(extra.end(), targets, targets + n_targets);
  std::vector<long long> first;
  for (size_t k = 0; k < prime_len; k++)
    if (prime[k] < V) first.push_back(-2 - (long long)k);
  if (first.empty()) {
    set_error("chunk_logits: empty prime");
    return CZ_ERR_INVALID;
  }
  GrowBuf &d_extra = m->sb[SB_EXTRA];
  CZ_TRY(d_extra.reserve(extra.size() * 4 + 16, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_extra.p, extra.data(), extra.size() * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  std::vector<RwUnit> units(1);
  build_unit(units[0], first, targets, n_targets, V, 0, [&](size_t q) { return -2 - (long long)(prime_len + q); });
  RwOut o;
  o.logits_host = logits_out;
  return rwkv_run_units(m, units, nullptr, d_extra.as<uint32_t>(), 0, o, 0, st);
}

// ---- lock-step batched decode (main.rs:2706-2864; gated hint primes as at 2803-2812, rebuilt from the decoded history) ---------
int rwkv_decode(cz_model *m, const uint8_t *payload, const uint64_t *seg_off, size_t n_tokens, const cz_schedule *sched, uint32_t *ids_out) {
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  const cz_model_config &c = m->cfg;
  const uint32_t S = sched->n_segments;
  const size_t V = c.vocab;
  uint64_t max_len = 0;
  for (uint32_t g = 0; g < S; g++) max_len = std::max<uint64_t>(max_len, sched->seg_start[g + 1] - sched->seg_start[g]);
  const size_t S_pad = (S + 3) & ~(size_t)3;
  GrowBuf &d_pay = m->sb[SB_PAY], &d_off = m->sb[SB_OFF], &d_start = m->sb[SB_START], &d_state = m->sb[SB_STATE], &d_ids = m->sb[SB_DIDS],
          &d_keep = m->sb[SB_LOGITS], &d_fresh = m->sb[SB_RW_FRESH], &d_meta = m->sb[SB_KVB];
  const uint64_t pay_total = seg_off[S];
  CZ_TRY(d_pay.reserve(pay_total + 16, st));
  CZ_TRY(d_off.reserve((S + 1) * 8, st));
  CZ_TRY(d_start.reserve((S + 1) * 8, st));
  CZ_TRY(d_state.reserve(S * decoder_state_bytes(), st));
  CZ_TRY(d_ids.reserve(n_tokens * 4, st));
  CZ_TRY(d_keep.reserve(V * S_pad * 4, st));
  CZ_TRY(d_fresh.reserve(V * S_pad * 4, st));
  CZ_TRY(d_meta.reserve(S * 4 * 8 + 64, st));
  CZ_TRY(ensure_workspace(m, S, S, 0));
  CZ_TRY(rwkv_ensure_ws(m, S, S));
  CZ_TRY(ensure_logits(m, S));
  CZ_TRY(digest_begin(m, n_tokens, S, st));
  Workspace &ws = m->ws;
  RwkvWs &rw = m->rws;
  int *d_active = d_meta.as<int>(), *d_cm_keep = d_active + S, *d_sym = d_cm_keep + S;
  CZ_CUDA_TRY(cudaMemcpyAsync(d_pay.p, payload, pay_total, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_off.p, seg_off, (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_start.p, sched->seg_start, (S + 1) * 8, cudaMemcpyHostToDevice, st));
  CZ_TRY(launch_decoder_init(ctx, d_pay.as<uint8_t>(), d_off.as<uint64_t>(), (int)S, d_state.p, st));
  MatchDecView mview;  // the match model's per-stream state: literal escapes are ordinary symbols to it (a hit on one steps nothing)
  if (m->match_order) CZ_TRY(match_decode_begin(m, S, n_tokens, st, &mview));
  const bool use_cm = c.engine == CZ_ENGINE_TCGEN05 && getenv("CZ_DEBUG_NO_COLMAX") == nullptr;
  const bool use_graph = getenv("CZ_DECODE_NO_GRAPH") == nullptr;
  unsigned long long *d_ctr = (unsigned long long *)(((uintptr_t)(d_sym + S) + 15) & ~(uintptr_t)15);  // aligned tail of d_meta
  const size_t total = V * S_pad;
  std::vector<int> iota(S), minus1(S, -1), ones(S, 1), next(S);
  for (uint32_t g = 0; g < S; g++) {
    iota[g] = (int)g;
    next[g] = (int)g + 1;
  }
  // head + commit of the freshly computed logits columns of the streams flagged in d_active
  auto head_commit = [&]() -> int {
    bool have_max = false;
    CZ_TRY(rwkv_final_norm_gather(m, (int)S, st));
    CZ_TRY(lm_head(m, 0, (int)S, d_fresh.as<float>(), S_pad, st, ws.colmax, &have_max));
    CZ_LAUNCH(ctx, CZ_K_OTHER,
              (czk::rw_commit_logits_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, st>>>(d_fresh.as<float>(), d_keep.as<float>(), S_pad, total,
                                                                                           d_active, have_max ? ws.colmax : nullptr, d_cm_keep, (int)S)));
    CZ_CHECK_LAUNCH();
    return CZ_OK;
  };
  // (re)start every stream from a zero state and feed `first` (BOS, or a gated hint prime: main.rs:2803-2812 ->
  // models.rs:162-170), leaving the logits of its last token in d_keep; then restore the single-row step metadata.  A long prime
  // goes in slabs of at most max_rows rows (the encoder's bound), the state carried from slab to slab, so the workspace does not
  // grow with the history; any split gives the same logits bit for bit (DESIGN §3).
  const size_t max_rows = sched->max_batch_tokens ? sched->max_batch_tokens : kSlabRows, Tw = std::max<size_t>(1, max_rows / S);
  // with a dictionary, the streams start from the state it leaves (rwkv_prefix: `first` is then its last in-vocabulary symbol)
  const RwPrefix prefix = rwkv_prefix(m, sched->bos);
  auto prime_all = [&](const std::vector<uint32_t> &first) -> int {
    const size_t n = first.size();
    CZ_CUDA_TRY(cudaMemcpyAsync(d_active, ones.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_TRY(rwkv_state_reset(m, m->rstate, S, st));
    CZ_TRY(rwkv_prefix_state(m, m->rstate, prefix, S, max_rows, st));
    for (size_t k0 = 0; k0 < n; k0 += Tw) {
      const size_t T = std::min(Tw, n - k0), R = (size_t)S * T;
      CZ_TRY(ensure_workspace(m, R, S, 0));
      CZ_TRY(rwkv_ensure_ws(m, R, S));
      std::vector<uint32_t> tok(R);
      std::vector<int> prev(R), slot(R), flags(R, 0), rb(S), re(S), lrows(S);
      for (uint32_t g = 0; g < S; g++) {
        for (size_t k = 0; k < T; k++) {
          const size_t r = (size_t)g * T + k;
          tok[r] = first[k0 + k];
          prev[r] = k == 0 ? -1 : (int)r - 1;
          slot[r] = (int)g;
        }
        flags[(size_t)g * T + T - 1] = 1;
        rb[g] = (int)(g * T);
        re[g] = (int)(g * T + T);
        lrows[g] = (int)(g * T + T - 1);
      }
      CZ_CUDA_TRY(cudaMemcpyAsync(ws.tok, tok.data(), R * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.prev_row, prev.data(), R * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.slot, slot.data(), R * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.flags, flags.data(), R * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_begin, rb.data(), S * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_end, re.data(), S * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(rw.stream_slot, iota.data(), S * 4, cudaMemcpyHostToDevice, st));
      CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, lrows.data(), S * 4, cudaMemcpyHostToDevice, st));
      CZ_TRY(rwkv_forward(m, (int)R, (int)S, m->rstate, /*in_place=*/n == 1, nullptr, st));
      if (k0 + T < n) CZ_CUDA_TRY(cudaStreamSynchronize(st));  // the staging vectors are stack-owned
    }
    CZ_TRY(head_commit());
    // single-row step metadata: row s = stream s, state slot s
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.prev_row, minus1.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.slot, iota.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.flags, ones.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_begin, iota.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_end, next.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, iota.data(), S * 4, cudaMemcpyHostToDevice, st));
    CZ_CUDA_TRY(cudaStreamSynchronize(st));  // the staging vectors are stack-owned
    return CZ_OK;
  };
  auto decode_syms = [&]() -> int {
    // f-4: digest of the logits column each live stream is about to decode from, at index seg_start[g] + ctr[0].  A stream that
    // decoded a literal escape did not step, so its kept column is the one the encoder coded the next symbol from.
    if (m->digest_host)
      CZ_TRY(launch_logits_digest(ctx, d_keep.as<float>(), V, S, S_pad, m->sb[SB_CV].p, m->sb[SB_DIGEST].as<uint8_t>(), 0, nullptr,
                                  d_start.as<uint64_t>(), d_ctr, st));
    return launch_decode_step(ctx, CZ_CDF_RWKV_LITERALS, d_keep.as<float>(), (int)V, S_pad, (int)S, d_pay.as<uint8_t>(), d_off.as<uint64_t>(),
                              d_start.as<uint64_t>(), 0, d_state.p, d_ids.as<uint32_t>(), (uint32_t *)d_sym, use_cm ? d_cm_keep : nullptr, st,
                              d_ctr, m->match_order ? &mview : nullptr);
  };
  // one step = decode a symbol per stream, decide which streams step (literals do not), single-token forward, commit the new
  // logits columns.  The step-varying scalar (coded index) lives in d_ctr, so the launch sequence is captured once into a CUDA
  // graph and replayed for the remaining steps.
  auto step = [&]() -> int {
    CZ_TRY(decode_syms());
    CZ_LAUNCH(ctx, CZ_K_OTHER,
              (czk::rw_decode_flags_kernel<<<(unsigned)ceil_div(S, 128), 128, 0, st>>>((const uint32_t *)d_sym, (uint32_t)V, d_start.as<uint64_t>(), d_ctr,
                                                                                      (int)S, rw.flags, d_active, ws.tok)));
    CZ_CHECK_LAUNCH();
    CZ_TRY(rwkv_forward(m, (int)S, (int)S, m->rstate, /*in_place=*/true, d_active, st));
    CZ_TRY(head_commit());
    CZ_TRY(launch_advance_ctr(ctx, d_ctr, st));
    return CZ_OK;
  };
  // units as the encoder plans them; each starts from a fresh state primed with BOS / the event's prime (events: S == 1)
  std::vector<RwCut> cut;
  CZ_TRY(rwkv_plan_units(sched, max_len, (uint32_t)V, cut));
  std::vector<uint32_t> extra, ids_host, first;  // explicit prime tokens of the events; decoded ids [0, n_host) of the one stream
  std::vector<size_t> ev_off(sched->n_events + 1, 0);
  for (uint32_t e = 0; e < sched->n_events; e++) {
    ev_off[e] = extra.size();
    extra.insert(extra.end(), sched->events[e].prime, sched->events[e].prime + sched->events[e].prime_len);
  }
  std::vector<long long> src;
  uint64_t n_host = 0;
  for (size_t u = 0; u < cut.size(); u++) {
    const uint64_t c0 = cut[u].begin, c1 = u + 1 < cut.size() ? cut[u + 1].begin : max_len;
    first.assign(1, prefix.last == -1 ? sched->bos : m->dictionary[(size_t)(-2 - prefix.last)]);
    if (cut[u].event >= 0) {
      const cz_prime_event &ev = sched->events[cut[u].event];
      if (ev.hist_take && n_host < c0) {  // the history tail needs what has been decoded so far on the host: one copy per event
        ids_host.resize(c0);
        CZ_CUDA_TRY(cudaMemcpyAsync(ids_host.data() + n_host, d_ids.as<uint32_t>() + n_host, (c0 - n_host) * 4, cudaMemcpyDeviceToHost, st));
        CZ_CUDA_TRY(cudaStreamSynchronize(st));
        n_host = c0;
      }
      rwkv_event_prime(ev, ids_host.data(), 0, c0, (uint32_t)V, ev_off[cut[u].event], src);
      first.resize(src.size());
      for (size_t k = 0; k < src.size(); k++) first[k] = src[k] >= 0 ? ids_host[src[k]] : (src[k] == -1 ? sched->bos : extra[-2 - src[k]]);
    }
    CZ_TRY(prime_all(first));
    CZ_TRY(launch_set_ctr(ctx, d_ctr, c0, 0, st));
    cudaGraphExec_t gexec = nullptr;
    uint64_t nodes = 0;
    int rc = CZ_OK;
    const uint64_t n_steps = c1 - c0 - (u + 1 == cut.size() ? 1 : 0);  // the very last symbol needs no step after it
    for (uint64_t i = 0; i < n_steps && rc == CZ_OK; i++) {
      if (i == 0 || !use_graph || n_steps < 4) {
        rc = step();
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
          set_error(std::string("rwkv decode step graph capture failed: ") + cudaGetErrorString(e));
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
      if (rc == CZ_OK && (i & 1023) == 1023) rc = fetch_device_status(ctx, nullptr, nullptr);
    }
    if (gexec) cudaGraphExecDestroy(gexec);
    CZ_TRY(rc);
  }
  CZ_TRY(decode_syms());  // every stream's last symbol
  CZ_TRY(fetch_device_status(ctx, nullptr, nullptr));
  CZ_CUDA_TRY(cudaMemcpyAsync(ids_out, d_ids.p, n_tokens * 4, cudaMemcpyDeviceToHost, st));
  CZ_TRY(digest_end(m, n_tokens, st));
  CZ_TRY(match_decode_end(m, n_tokens, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  return CZ_OK;
}

// ---- batch-of-1 session shim (Rwkv7Session, src/models.rs:151-179) --------------------------------------------------------------
int rwkv_session_forward(cz_model *m, RwkvState &stt, const uint32_t *tok, size_t n, bool reset, float *logits_dev4, float *logits_out) {
  cz_ctx *ctx = m->ctx;
  cudaStream_t st = ctx->stream;
  CZ_TRY(ensure_workspace(m, n, 1, 0));
  CZ_TRY(rwkv_ensure_ws(m, n, 1));
  if (reset || stt.cap == 0) CZ_TRY(rwkv_state_reset(m, stt, 1, st));
  Workspace &ws = m->ws;
  RwkvWs &rw = m->rws;
  std::vector<int> prev(n), slot(n, 0), flags(n, 0);
  for (size_t i = 0; i < n; i++) prev[i] = (int)i - 1;
  flags[n - 1] = 1;
  const int rb = 0, re = (int)n, sl = 0, lrow = (int)n - 1;
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.tok, tok, n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.prev_row, prev.data(), n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.slot, slot.data(), n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.flags, flags.data(), n * 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_begin, &rb, 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.row_end, &re, 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(rw.stream_slot, &sl, 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaMemcpyAsync(ws.logit_rows, &lrow, 4, cudaMemcpyHostToDevice, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  CZ_TRY(rwkv_forward(m, (int)n, 1, stt, /*in_place=*/n == 1, nullptr, st));
  CZ_TRY(rwkv_final_norm_gather(m, 1, st));
  CZ_TRY(lm_head(m, 0, 1, logits_dev4, 4, st));
  CZ_CUDA_TRY(cudaMemcpy2DAsync(logits_out, 4, logits_dev4, 16, 4, (size_t)m->cfg.vocab, cudaMemcpyDeviceToHost, st));
  CZ_CUDA_TRY(cudaStreamSynchronize(st));
  return CZ_OK;
}

}  // namespace cz
