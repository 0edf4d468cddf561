// Match model (cz_model_set_match, DESIGN.md §6): a token whose last K symbols repeat those before an earlier position of its segment is
// predicted to be the symbol that followed there; the prediction is coded as a binary flag interval (total 2^30) in front of the
// model's interval, and a hit's model interval is not coded at all.
//
// Encode runs over every coded token of a call at once, after the model's intervals are known:
//   match_hash_kernel       context key of every position (segment-relative position >= K), and its segment
//   cub::DeviceRadixSort    keys key << 40 | global index: equal keys end up adjacent, in index order
//   match_find_kernel       the sorted predecessor with the same key is the candidate j(i) if it lies in i's segment; verify and
//                           length (how far the contexts agree, up to K + 15), the prediction and its bucket
//   match_tile_kernel       per tile of 1,024 tokens: segmented per-bucket counts of tries and hits, and the number of misses
//   match_tile_scan_kernel  carries of those counts from tile to tile (reset at segment starts), and the misses' offsets
//   match_weight_kernel     per token: the exclusive counts of its bucket in its segment -> W; its place in the interval list
//   match_assemble_kernel   the interval list (flag, then the model's interval unless it was a hit) and the lanes' offsets in it
// Decode keeps the same state per stream and advances it inside the captured decode step (exec.cu, decode_step_kernel).
#include <cub/device/device_radix_sort.cuh>

#include "match.h"

namespace czk {

using cz::kMatchBuckets;
using cz::kMatchHashBits;
using cz::kMatchNone;

constexpr int MT_TILE = 1024;  // tokens per tile of the counting passes (one CTA, one token per thread)
constexpr uint32_t MI_HAS = 1u << 31, MI_HIT = 1u << 30;  // info word: has a prediction, it was right; bucket in the low bits
constexpr uint64_t IDX_MASK = (1ull << 40) - 1;

// key(i) over t[i-K .. i-1], oldest first (FNV-1a over u32 symbols, then a Fibonacci hash to HB bits)
__device__ __forceinline__ uint32_t match_key(const uint32_t *t, int K) {
  uint32_t h = 0x811C9DC5u;
  for (int k = 0; k < K; k++) h = (h ^ t[k]) * 0x01000193u;
  return (h * 0x9E3779B1u) >> (32 - kMatchHashBits);
}

__device__ __forceinline__ uint32_t match_weight(uint32_t hits, uint32_t tries) {
  uint64_t p = ((2ull * hits + 1) << 16) / (2ull * tries + 2);
  p = p < 1 ? 1 : (p > 65535 ? 65535 : p);
  return (uint32_t)p << 14;
}

// segment of global index i: the last g with seg_start[g] <= i (empty segments share a start; i < seg_start[S] = n)
__device__ __forceinline__ uint32_t segment_of(const uint64_t *seg_start, uint32_t S, uint64_t i) {
  uint32_t lo = 0, hi = S;  // seg_start[lo] <= i < seg_start[hi]
  while (lo + 1 < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (seg_start[mid] <= i) lo = mid;
    else hi = mid;
  }
  return lo;
}

__global__ void match_hash_kernel(const uint32_t *__restrict__ ids, const uint64_t *__restrict__ seg_start, uint32_t S, uint64_t n, int K,
                                  uint32_t *__restrict__ sid, unsigned long long *__restrict__ keys) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t g = segment_of(seg_start, S, i);
  sid[i] = g;
  const uint64_t key = i - seg_start[g] >= (uint64_t)K ? match_key(ids + i - K, K) : (1u << kMatchHashBits);  // sentinel: no context
  keys[i] = (key << 40) | i;
}

__global__ void match_find_kernel(const unsigned long long *__restrict__ sorted, const uint32_t *__restrict__ ids,
                                  const uint32_t *__restrict__ sid, const uint64_t *__restrict__ seg_start, uint64_t n, int K,
                                  uint32_t *__restrict__ pred, uint32_t *__restrict__ info) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const uint64_t e = sorted[r], i = e & IDX_MASK, key = e >> 40;
  uint32_t pr = kMatchNone, inf = 0;
  if (key < (1u << kMatchHashBits) && r > 0 && (sorted[r - 1] >> 40) == key) {
    const uint64_t j = sorted[r - 1] & IDX_MASK;  // the most recent earlier position with the same key, in any segment
    const uint32_t g = sid[i];
    if (sid[j] == g) {
      const uint64_t s0 = seg_start[g];
      const uint32_t cap = (uint32_t)K + kMatchBuckets - 1;
      uint32_t len = 0;
      while (len < cap && j - len > s0 && ids[j - 1 - len] == ids[i - 1 - len]) len++;
      if (len >= (uint32_t)K) {  // (shorter: a hash collision, no prediction)
        pr = ids[j];
        inf = MI_HAS | (ids[i] == pr ? MI_HIT : 0u) | (len - (uint32_t)K);
      }
    }
  }
  pred[i] = pr;
  info[i] = inf;
}

// Per-warp summary of 32 consecutive tokens for the segmented counts: f / l = segment of the first / last token, agg[c] (one counter
// per lane: tries of bucket c for c < 16, hits of bucket c - 16 above) over the tokens of segment l only, misses over all of them.
// Groups combine left to right with  state (sid, cnt) + group (f, l, agg):  carry into the group = f == sid ? cnt : 0;
// new state = (l, (l == sid ? cnt : 0) + agg)  -- segment ids never decrease along the tokens.
struct WarpSum {
  uint32_t f, l, agg, miss;
};
__device__ __forceinline__ WarpSum warp_summary(uint32_t s, uint32_t inf) {
  const int lane = threadIdx.x & 31;
  WarpSum w;
  w.f = __shfl_sync(0xffffffffu, s, 0);
  w.l = __shfl_sync(0xffffffffu, s, 31);
  const bool in_l = s == w.l && (inf & MI_HAS);
  const uint32_t b = inf & 31u;
  w.agg = 0;
#pragma unroll
  for (int c = 0; c < 32; c++) {
    const bool p = in_l && b == (uint32_t)(c & 15) && (c < 16 || (inf & MI_HIT));
    const uint32_t bal = __ballot_sync(0xffffffffu, p);
    if (lane == c) w.agg = __popc(bal);
  }
  w.miss = __popc(__ballot_sync(0xffffffffu, (inf & MI_HAS) && !(inf & MI_HIT)));
  return w;
}

// token of thread i of the tile: tokens past n act as a token of the last segment without a prediction
__device__ __forceinline__ void load_token(const uint32_t *sid, const uint32_t *info, uint64_t n, uint64_t i, uint32_t &s, uint32_t &inf) {
  if (i < n) {
    s = sid[i];
    inf = info[i];
  } else {
    s = sid[n - 1];
    inf = 0;
  }
}

__global__ void __launch_bounds__(MT_TILE) match_tile_kernel(const uint32_t *__restrict__ sid, const uint32_t *__restrict__ info, uint64_t n,
                                                            uint32_t *__restrict__ tile_fl, uint32_t *__restrict__ tile_agg,
                                                            uint32_t *__restrict__ tile_miss) {
  __shared__ uint32_t s_f[32], s_l[32], s_agg[32][32], s_miss[32];
  const uint64_t i = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t s, inf;
  load_token(sid, info, n, i, s, inf);
  const WarpSum w = warp_summary(s, inf);
  if (lane == 0) {
    s_f[warp] = w.f;
    s_l[warp] = w.l;
    s_miss[warp] = w.miss;
  }
  s_agg[warp][lane] = w.agg;
  __syncthreads();
  if (warp == 0) {
    uint32_t cur = s_f[0], cnt = 0, miss = 0;
    for (int v = 0; v < 32; v++) {
      cnt = (s_l[v] == cur ? cnt : 0u) + s_agg[v][lane];
      cur = s_l[v];
      miss += s_miss[v];
    }
    tile_agg[(size_t)blockIdx.x * 32 + lane] = cnt;
    if (lane == 0) {
      tile_fl[2 * blockIdx.x] = s_f[0];
      tile_fl[2 * blockIdx.x + 1] = s_l[31];
      tile_miss[blockIdx.x] = miss;
    }
  }
}

// one warp: lane c carries counter c across the tiles in order; lane 0 also the misses (not segmented)
__global__ void match_tile_scan_kernel(const uint32_t *__restrict__ tile_fl, const uint32_t *__restrict__ tile_agg,
                                       const uint32_t *__restrict__ tile_miss, uint32_t n_tiles, uint32_t *__restrict__ tile_carry,
                                       unsigned long long *__restrict__ tile_moff) {
  const int lane = threadIdx.x;
  uint32_t cur = tile_fl[0], cnt = 0;
  unsigned long long moff = 0;
#pragma unroll 4
  for (uint32_t t = 0; t < n_tiles; t++) {
    const uint32_t f = tile_fl[2 * t], l = tile_fl[2 * t + 1], a = tile_agg[(size_t)t * 32 + lane];
    tile_carry[(size_t)t * 32 + lane] = f == cur ? cnt : 0u;
    cnt = (l == cur ? cnt : 0u) + a;
    cur = l;
    if (lane == 0) {
      tile_moff[t] = moff;
      moff += tile_miss[t];
    }
  }
}

__global__ void __launch_bounds__(MT_TILE) match_weight_kernel(const uint32_t *__restrict__ sid, const uint32_t *__restrict__ info, uint64_t n,
                                                              const uint32_t *__restrict__ tile_fl, const uint32_t *__restrict__ tile_carry,
                                                              const unsigned long long *__restrict__ tile_moff, uint32_t *__restrict__ wout,
                                                              unsigned long long *__restrict__ list_pos) {
  __shared__ uint32_t s_f[32], s_l[32], s_agg[32][32], s_miss[32];
  __shared__ uint32_t s_carry[32][32], s_moff[32];
  const uint64_t i = (uint64_t)blockIdx.x * MT_TILE + threadIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t s, inf;
  load_token(sid, info, n, i, s, inf);
  const WarpSum w = warp_summary(s, inf);
  if (lane == 0) {
    s_f[warp] = w.f;
    s_l[warp] = w.l;
    s_miss[warp] = w.miss;
  }
  s_agg[warp][lane] = w.agg;
  __syncthreads();
  if (warp == 0) {  // carries into every warp, for the segment of its first token
    uint32_t cur = tile_fl[2 * blockIdx.x], cnt = tile_carry[(size_t)blockIdx.x * 32 + lane], miss = 0;
    for (int v = 0; v < 32; v++) {
      s_carry[v][lane] = s_f[v] == cur ? cnt : 0u;
      cnt = (s_l[v] == cur ? cnt : 0u) + s_agg[v][lane];
      cur = s_l[v];
      if (lane == 0) {
        s_moff[v] = miss;
        miss += s_miss[v];
      }
    }
  }
  __syncthreads();
  const uint32_t lt = (1u << lane) - 1u;
  const bool has = inf & MI_HAS, hit = inf & MI_HIT, miss = has && !hit;
  const uint32_t b = inf & 31u;
  // lanes before this one with the same segment and the same bucket (tokens without a prediction form a group of their own)
  const uint32_t same = has ? __match_any_sync(0xffffffffu, ((unsigned long long)s << 5) | b) : (__match_any_sync(0xffffffffu, ~0ull), 0u);
  const uint32_t hits_bal = __ballot_sync(0xffffffffu, hit), miss_bal = __ballot_sync(0xffffffffu, miss);
  if (i >= n) return;
  uint32_t W = 0;
  if (has) {
    const bool carried = s == s_f[warp];
    const uint32_t tries = (carried ? s_carry[warp][b] : 0u) + __popc(same & lt);
    const uint32_t hits = (carried ? s_carry[warp][16 + b] : 0u) + __popc(same & hits_bal & lt);
    W = match_weight(hits, tries);
  }
  wout[i] = W;
  const unsigned long long p = i + tile_moff[blockIdx.x] + s_moff[warp] + __popc(miss_bal & lt);
  list_pos[i] = p;
  if (i == n - 1) list_pos[n] = p + 1 + (miss ? 1 : 0);
}

__global__ void match_assemble_kernel(const uint32_t *__restrict__ c_lo, const uint32_t *__restrict__ c_hi, const uint32_t *__restrict__ info,
                                      const uint32_t *__restrict__ wt, const unsigned long long *__restrict__ list_pos, uint64_t n,
                                      const uint64_t *__restrict__ seg_start, uint32_t S, uint32_t *__restrict__ list_lo,
                                      uint32_t *__restrict__ list_hi, uint64_t *__restrict__ lane_off) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i <= S) lane_off[i] = list_pos[seg_start[i]];
  if (i >= n) return;
  uint64_t p = list_pos[i];
  const uint32_t inf = info[i];
  if (inf & MI_HAS) {
    const uint32_t W = wt[i];
    const bool hit = inf & MI_HIT;
    list_lo[p] = hit ? 0u : W;
    list_hi[p] = hit ? W : CZ_AC_CDF_TOTAL;
    if (hit) return;
    p++;
  }
  list_lo[p] = c_lo[i];
  list_hi[p] = c_hi[i];
}

// list index -> coded-token index: the last token of [a, b) whose first interval sits at or before list index L.  A flag interval is
// never empty (W in [2^14, 2^30 - 2^14]), so a zero-width interval is always the model interval of that token.
__device__ __forceinline__ uint64_t token_of_list_index(const unsigned long long *list_pos, uint64_t a, uint64_t b, uint64_t L) {
  while (a + 1 < b) {
    const uint64_t mid = (a + b) >> 1;
    if (list_pos[mid] <= L) a = mid;
    else b = mid;
  }
  return a;
}
__global__ void match_zw_map_kernel(const unsigned long long *__restrict__ list_pos, const uint64_t *__restrict__ seg_start,
                                    const uint64_t *__restrict__ list_lane_off, uint32_t S, uint64_t n, unsigned long long *__restrict__ lane_zw,
                                    unsigned long long *__restrict__ err_index) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < S && lane_zw && lane_zw[g] != ~0ull)
    lane_zw[g] = token_of_list_index(list_pos, seg_start[g], seg_start[g + 1], list_lane_off[g] + lane_zw[g]) - seg_start[g];
  if (g == S && *err_index != ~0ull) *err_index = token_of_list_index(list_pos, 0, n, *err_index);
}

}  // namespace czk

namespace cz {

// layout of the encode scratch (SB_MATCH) for n tokens, S segments
struct MatchEncBufs {
  unsigned long long *keys_in, *keys_out, *list_pos, *tile_moff;
  uint64_t *lane_off;
  uint32_t *sid, *pred, *info, *w, *list_lo, *list_hi, *tile_fl, *tile_agg, *tile_carry, *tile_miss;
  size_t bytes;
};
static MatchEncBufs match_enc_layout(void *base, size_t n, uint32_t S) {
  const size_t T = ceil_div(n, czk::MT_TILE);
  MatchEncBufs b;
  char *p = (char *)base;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char *q = p + off;
    off += (bytes + 255) & ~(size_t)255;
    return (void *)q;
  };
  b.keys_in = (unsigned long long *)take(n * 8);
  b.keys_out = (unsigned long long *)take(n * 8);
  b.list_pos = (unsigned long long *)take((n + 1) * 8);
  b.tile_moff = (unsigned long long *)take(T * 8);
  b.lane_off = (uint64_t *)take((S + 1) * 8);
  b.sid = (uint32_t *)take(n * 4);
  b.pred = (uint32_t *)take(n * 4);
  b.info = (uint32_t *)take(n * 4);
  b.w = (uint32_t *)take(n * 4);
  b.list_lo = (uint32_t *)take(2 * n * 4);
  b.list_hi = (uint32_t *)take(2 * n * 4);
  b.tile_fl = (uint32_t *)take(T * 8);
  b.tile_agg = (uint32_t *)take(T * 32 * 4);
  b.tile_carry = (uint32_t *)take(T * 32 * 4);
  b.tile_miss = (uint32_t *)take(T * 4);
  b.bytes = off;
  return b;
}

int match_encode_intervals(cz_model *m, const uint32_t *ids_dev, size_t n, const uint64_t *seg_start_dev, uint32_t S, const uint32_t *c_lo_dev,
                           const uint32_t *c_hi_dev, cudaStream_t st, const uint32_t **list_lo, const uint32_t **list_hi,
                           const uint64_t **list_lane_off) {
  cz_ctx *ctx = m->ctx;
  const int K = (int)m->match_order;
  const size_t T = ceil_div(n, czk::MT_TILE);
  GrowBuf &buf = m->sb[SB_MATCH], &tmp = m->sb[SB_MTEMP];
  CZ_TRY(buf.reserve(match_enc_layout(nullptr, n, S).bytes + 256, st));
  const MatchEncBufs b = match_enc_layout(buf.p, n, S);
  const int end_bit = 40 + kMatchHashBits + 1;
  size_t tmp_bytes = 0;
  CZ_CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, b.keys_in, b.keys_out, (int64_t)n, 0, end_bit, st));
  CZ_TRY(tmp.reserve(tmp_bytes + 16, st));
  const unsigned grid = (unsigned)ceil_div(n, 256);
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::match_hash_kernel<<<grid, 256, 0, st>>>(ids_dev, seg_start_dev, S, n, K, b.sid, b.keys_in)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            CZ_CUDA_TRY(cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, b.keys_in, b.keys_out, (int64_t)n, 0, end_bit, st)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::match_find_kernel<<<grid, 256, 0, st>>>(b.keys_out, ids_dev, b.sid, seg_start_dev, n, K, b.pred, b.info)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::match_tile_kernel<<<(unsigned)T, czk::MT_TILE, 0, st>>>(b.sid, b.info, n, b.tile_fl, b.tile_agg, b.tile_miss)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::match_tile_scan_kernel<<<1, 32, 0, st>>>(b.tile_fl, b.tile_agg, b.tile_miss, (uint32_t)T, b.tile_carry, b.tile_moff)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_OTHER,
            (czk::match_weight_kernel<<<(unsigned)T, czk::MT_TILE, 0, st>>>(b.sid, b.info, n, b.tile_fl, b.tile_carry, b.tile_moff, b.w,
                                                                          b.list_pos)));
  CZ_CHECK_LAUNCH();
  CZ_LAUNCH(ctx, CZ_K_CODER,
            (czk::match_assemble_kernel<<<(unsigned)ceil_div(std::max<size_t>(n, (size_t)S + 1), 256), 256, 0, st>>>(
                c_lo_dev, c_hi_dev, b.info, b.w, b.list_pos, n, seg_start_dev, S, b.list_lo, b.list_hi, b.lane_off)));
  CZ_CHECK_LAUNCH();
  *list_lo = b.list_lo;
  *list_hi = b.list_hi;
  *list_lane_off = b.lane_off;
  return CZ_OK;
}

int match_encode_finish(cz_model *m, size_t n, const uint64_t *seg_start_dev, uint32_t S, unsigned long long *lane_zw_dev,
                        unsigned long long *err_index_dev, cudaStream_t st) {
  const MatchEncBufs b = match_enc_layout(m->sb[SB_MATCH].p, n, S);
  CZ_LAUNCH(m->ctx, CZ_K_CODER,
            (czk::match_zw_map_kernel<<<(unsigned)ceil_div((size_t)S + 1, 128), 128, 0, st>>>(b.list_pos, seg_start_dev, b.lane_off, S, n,
                                                                                             lane_zw_dev, err_index_dev)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

int match_encode_copy_out(cz_model *m, size_t n, uint32_t S, cudaStream_t st) {
  if (!n || (!m->mo_pred_host && !m->mo_w_host)) return CZ_OK;
  const MatchEncBufs b = match_enc_layout(m->sb[SB_MATCH].p, n, S);
  if (m->mo_pred_host) CZ_CUDA_TRY(cudaMemcpyAsync(m->mo_pred_host, b.pred, n * 4, cudaMemcpyDeviceToHost, st));
  if (m->mo_w_host) CZ_CUDA_TRY(cudaMemcpyAsync(m->mo_w_host, b.w, n * 4, cudaMemcpyDeviceToHost, st));
  return CZ_OK;
}

int match_decode_begin(cz_model *m, uint32_t S, size_t n_tokens, cudaStream_t st, MatchDecView *v) {
  const size_t tab = (size_t)S << kMatchHashBits, cnt = (size_t)S * 32, nxt = (size_t)S * 4;
  GrowBuf &d = m->sb[SB_MDEC];
  CZ_TRY(d.reserve((tab + cnt + nxt) * 4, st));
  v->table = d.as<uint32_t>();
  v->cnt = v->table + tab;
  v->next = v->cnt + cnt;
  v->order = m->match_order;
  CZ_CUDA_TRY(cudaMemsetAsync(v->table, 0, (tab + cnt) * 4, st));
  CZ_CUDA_TRY(cudaMemsetAsync(v->next, 0xFF, nxt * 4, st));  // pred = kMatchNone: position 0 < K has no prediction
  v->pred_out = v->w_out = nullptr;
  if (m->mo_pred_host || m->mo_w_host) {
    CZ_TRY(m->sb[SB_MOUT].reserve(n_tokens * 8 + 16, st));
    v->pred_out = m->sb[SB_MOUT].as<uint32_t>();
    v->w_out = v->pred_out + n_tokens;
  }
  return CZ_OK;
}

int match_decode_end(cz_model *m, size_t n_tokens, cudaStream_t st) {
  if (!n_tokens || !m->match_order || (!m->mo_pred_host && !m->mo_w_host)) return CZ_OK;
  const uint32_t *p = m->sb[SB_MOUT].as<uint32_t>();
  if (m->mo_pred_host) CZ_CUDA_TRY(cudaMemcpyAsync(m->mo_pred_host, p, n_tokens * 4, cudaMemcpyDeviceToHost, st));
  if (m->mo_w_host) CZ_CUDA_TRY(cudaMemcpyAsync(m->mo_w_host, p + n_tokens, n_tokens * 4, cudaMemcpyDeviceToHost, st));
  return CZ_OK;
}

}  // namespace cz
