// K7 / K8: RWKV-7 ("Goose") batched multi-stream forward for sm_100a.
//
// Replaces Rwkv7Session (src/models.rs:124-180) -> candle_rwkv7 Model::forward t==1 path
// (candle_rwkv7/src/models/rwkv7.rs:179-328 attention, 412-430 feed-forward, 468-478 block, 509-524 model, 529-542 group norm).
// The reference runs one token of one stream at a time through dozens of tiny candle ops.  Here a SLAB is
// [n_streams x T] token rows (stream-major, rows of one stream consecutive in time):
//   * everything that is not recurrent (LayerNorm, token-shift mixes, the r/k/v/o and FFN projections, the four LoRA pairs,
//     the LM head) runs over all rows at once: the dense contractions go through the tcgen05 GEMM (gemm_tcgen05.cu), with
//     tanh / sigmoid / relu^2 fused into its epilogues;
//   * the WKV-7 state recurrence  S <- S diag(w) - (S k^)(k^ (.) a)^T + v k~^T,  y = S r  runs in ONE kernel per layer: a warp
//     owns the 64x64 fp32 state of one (stream, head) in registers and walks the stream's rows in time order, with the per-token
//     prologue (decay, in-context learning rate a, value residual, k^ normalisation, k~) and epilogue (group norm eps 64e-5,
//     (r.k~.r_k) v bonus, gate) fused in, so the state is read and written once per slab, not once per token.
// ROW INVARIANCE (decode safety): the same kernels serve T-token slabs (encode) and T = 1 (stepwise decode); per-row arithmetic
// has a fixed order (per-lane sequential partials + fixed xor-shuffle trees, sequential j loops in the scan), so the logits of a
// (stream, position) do not depend on slab shape, batch size or GPU count.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "gemm.h"
#include "llama_kernels.h"
#include "model.h"

namespace czk {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int RW_MAXC = 1024;  // d_model <= 1024 (32 elements per lane)

// LayerNorm of one row by one warp: lane owns elements lane + 32*k.  Population variance, like candle's LayerNorm.
__device__ __forceinline__ void warp_layer_norm(const float *__restrict__ xr, const float *__restrict__ w, const float *__restrict__ b,
                                                int C, float eps, int lane, float (&out)[RW_MAXC / 32]) {
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++) {
    const int i = lane + 32 * k;
    out[k] = i < C ? xr[i] : 0.f;
    s += out[k];
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++) {
    const int i = lane + 32 * k;
    const float c = i < C ? out[k] - mean : 0.f;
    out[k] = c;
    q = fmaf(c, c, q);
  }
  const float inv = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++) {
    const int i = lane + 32 * k;
    if (i < C) out[k] = out[k] * inv * w[i] + b[i];
  }
}

// in-place LayerNorm of every row (layer 0 pre_norm, rwkv7.rs:470-472)
__global__ void __launch_bounds__(128) rwkv_ln_inplace_kernel(float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ b,
                                                              int n_rows, int C, float eps) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  float v[RW_MAXC / 32];
  warp_layer_norm(x + (size_t)row * C, w, b, C, eps, lane, v);
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++)
    if (lane + 32 * k < C) x[(size_t)row * C + lane + 32 * k] = v[k];
}

// LayerNorm + token shift + NMIX mixes (rwkv7.rs:185-201 with NMIX = 6; 414-424 with NMIX = 1):
//   xn = LN(x[row]);  prev = prev_row[row] >= 0 ? LN(x[prev_row[row]]) : state_in[slot[row]];  out_q = bf16(xn + (prev - xn) * mu_q)
// and, for the last row of a stream in this slab, state_out[slot] = xn (rwkv7.rs:306, 428).
// flags[row]: bit0 = last row of its stream in the slab, bit1 = row is inactive (stepwise decode: the stream just decoded a
// literal symbol and does not step, src/main.rs:2832-2834) -> no state write.
struct MixOut {
  __nv_bfloat16 *p[6];
};
struct MixMu {
  const float *p[6];
};
template <int NMIX>
__global__ void __launch_bounds__(128) rwkv_ln_mix_kernel(const float *__restrict__ x, const float *__restrict__ lnw,
                                                          const float *__restrict__ lnb, MixMu mu, const int *__restrict__ prev_row,
                                                          const int *__restrict__ slot, const int *__restrict__ flags,
                                                          const float *__restrict__ state_in, float *__restrict__ state_out,
                                                          MixOut out, int n_rows, int C, float eps) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  float xn[RW_MAXC / 32], pv[RW_MAXC / 32];
  warp_layer_norm(x + (size_t)row * C, lnw, lnb, C, eps, lane, xn);
  const int pr = prev_row[row], sl = slot[row], fl = flags[row];
  if (pr >= 0) {
    warp_layer_norm(x + (size_t)pr * C, lnw, lnb, C, eps, lane, pv);
  } else {
#pragma unroll
    for (int k = 0; k < RW_MAXC / 32; k++) pv[k] = lane + 32 * k < C ? state_in[(size_t)sl * C + lane + 32 * k] : 0.f;
  }
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++) {
    const int i = lane + 32 * k;
    if (i >= C) continue;
    const float xx = pv[k] - xn[k];
#pragma unroll
    for (int q = 0; q < NMIX; q++) out.p[q][(size_t)row * C + i] = __float2bfloat16_rn(xn[k] + xx * mu.p[q][i]);
    if ((fl & 1) && !(fl & 2)) state_out[(size_t)sl * C + i] = xn[k];
  }
}

// The same operator with 8 CONTIGUOUS elements per lane and chunk (C = NCH * 256: the 0.1B model's 768 = 3 chunks): 16-byte loads
// and 16-byte bf16 stores.  The element-per-lane form above issues 24 four-byte loads per operand and 144 two-byte stores per row
// for NMIX = 6 and moved 1.3 TB/s (ncu, profiles/ncu_summary_r02.md: issue 23%, 8.4 long-scoreboard stalls per issue); this one
// issues 6 + 18.  (Different lane -> element assignment, so the LayerNorm sums round differently: a model width takes one form or
// the other for good, encode and decode alike.)
template <int NCH>
__device__ __forceinline__ void warp_layer_norm_v8(const float *__restrict__ xr, const float *__restrict__ w, const float *__restrict__ b,
                                                   float eps, int lane, float (&out)[NCH][8]) {
  constexpr int C = NCH * 256;
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < NCH; c++) {
    const float4 *src = reinterpret_cast<const float4 *>(xr + (c * 32 + lane) * 8);
    const float4 a = src[0], d = src[1];
    out[c][0] = a.x; out[c][1] = a.y; out[c][2] = a.z; out[c][3] = a.w;
    out[c][4] = d.x; out[c][5] = d.y; out[c][6] = d.z; out[c][7] = d.w;
#pragma unroll
    for (int j = 0; j < 8; j++) s += out[c][j];
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < NCH; c++)
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float d = out[c][j] - mean;
      out[c][j] = d;
      q = fmaf(d, d, q);
    }
  const float inv = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
#pragma unroll
  for (int c = 0; c < NCH; c++) {
    const float4 *wp = reinterpret_cast<const float4 *>(w + (c * 32 + lane) * 8), *bp = reinterpret_cast<const float4 *>(b + (c * 32 + lane) * 8);
    const float4 w0 = __ldg(wp), w1 = __ldg(wp + 1), b0 = __ldg(bp), b1 = __ldg(bp + 1);
    const float ww[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w}, bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; j++) out[c][j] = out[c][j] * inv * ww[j] + bb[j];
  }
}

template <int NMIX, int NCH>
__global__ void __launch_bounds__(128) rwkv_ln_mix_v8_kernel(const float *__restrict__ x, const float *__restrict__ lnw,
                                                             const float *__restrict__ lnb, MixMu mu, const int *__restrict__ prev_row,
                                                             const int *__restrict__ slot, const int *__restrict__ flags,
                                                             const float *__restrict__ state_in, float *__restrict__ state_out,
                                                             MixOut out, int n_rows, float eps) {
  constexpr int C = NCH * 256;
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  float xn[NCH][8], pv[NCH][8];
  warp_layer_norm_v8<NCH>(x + (size_t)row * C, lnw, lnb, eps, lane, xn);
  const int pr = prev_row[row], sl = slot[row], fl = flags[row];
  if (pr >= 0) {
    warp_layer_norm_v8<NCH>(x + (size_t)pr * C, lnw, lnb, eps, lane, pv);
  } else {
#pragma unroll
    for (int c = 0; c < NCH; c++) {
      const float4 *src = reinterpret_cast<const float4 *>(state_in + (size_t)sl * C + (c * 32 + lane) * 8);
      const float4 a = src[0], d = src[1];
      pv[c][0] = a.x; pv[c][1] = a.y; pv[c][2] = a.z; pv[c][3] = a.w;
      pv[c][4] = d.x; pv[c][5] = d.y; pv[c][6] = d.z; pv[c][7] = d.w;
    }
  }
#pragma unroll
  for (int c = 0; c < NCH; c++) {
    const int base = (c * 32 + lane) * 8;
    float xx[8];
#pragma unroll
    for (int j = 0; j < 8; j++) xx[j] = pv[c][j] - xn[c][j];
#pragma unroll
    for (int q = 0; q < NMIX; q++) {
      const float4 *mp = reinterpret_cast<const float4 *>(mu.p[q] + base);
      const float4 m0 = __ldg(mp), m1 = __ldg(mp + 1);
      const float mm[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(xn[c][j] + xx[j] * mm[j], xn[c][j + 1] + xx[j + 1] * mm[j + 1]);
        pk[j >> 1] = *reinterpret_cast<const uint32_t *>(&h);
      }
      *reinterpret_cast<uint4 *>(out.p[q] + (size_t)row * C + base) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
    if ((fl & 1) && !(fl & 2)) {
      float4 *dst = reinterpret_cast<float4 *>(state_out + (size_t)sl * C + base);
      dst[0] = make_float4(xn[c][0], xn[c][1], xn[c][2], xn[c][3]);
      dst[1] = make_float4(xn[c][4], xn[c][5], xn[c][6], xn[c][7]);
    }
  }
}

// final LayerNorm of the gathered logit rows -> bf16 (rwkv7.rs:515)
__global__ void __launch_bounds__(128) rwkv_ln_gather_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                             const float *__restrict__ b, const int *__restrict__ rows,
                                                             __nv_bfloat16 *__restrict__ y, int n_out, int C, float eps) {
  const int j = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= n_out) return;
  float v[RW_MAXC / 32];
  warp_layer_norm(x + (size_t)rows[j] * C, w, b, C, eps, lane, v);
#pragma unroll
  for (int k = 0; k < RW_MAXC / 32; k++)
    if (lane + 32 * k < C) y[(size_t)j * C + lane + 32 * k] = __float2bfloat16_rn(v[k]);
}

// ---- the WKV-7 scan -------------------------------------------------------------------------------------------------------
// One warp per (stream, head).  Lane l owns state rows i0 = l and i1 = l + 32 (64 fp32 each, in registers).
// State layout in HBM (internal): S[(j/4) * 64 + i] as float4 over j%4  -> a warp's loads/stores are 512 contiguous bytes.
struct WkvVecs {  // per-layer fp32 vectors, each [C]
  const float *w0, *a0, *v0, *k_k, *k_a, *r_k, *gn_w, *gn_b;
};
struct WkvIo {  // per-row fp32 GEMM outputs [R][C]
  const float *r, *k, *v, *wl, *al, *vl, *g;
  float *v_first;  // layer 0 writes it, layers > 0 read it
};

__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

template <bool LAYER0>
__global__ void __launch_bounds__(32) wkv7_scan_kernel(WkvIo io, WkvVecs vc, const int *__restrict__ row_begin,
                                                       const int *__restrict__ row_end, const int *__restrict__ stream_slot,
                                                       const int *__restrict__ stream_active, float *__restrict__ state,
                                                       __nv_bfloat16 *__restrict__ out, int C, int H) {
  __shared__ __align__(16) float s_w[64], s_kk[64], s_ka[64], s_kp[64], s_r[64];
  const int s = blockIdx.x, h = blockIdx.y, lane = threadIdx.x;
  if (stream_active && !stream_active[s]) return;
  const int rb = row_begin[s], re = row_end[s];
  if (rb >= re) return;
  float4 *st4 = reinterpret_cast<float4 *>(state + ((size_t)stream_slot[s] * H + h) * 4096);
  float S0[64], S1[64];
#pragma unroll
  for (int j4 = 0; j4 < 16; j4++) {
    const float4 a = st4[j4 * 64 + lane], b = st4[j4 * 64 + lane + 32];
    S0[4 * j4] = a.x; S0[4 * j4 + 1] = a.y; S0[4 * j4 + 2] = a.z; S0[4 * j4 + 3] = a.w;
    S1[4 * j4] = b.x; S1[4 * j4 + 1] = b.y; S1[4 * j4 + 2] = b.z; S1[4 * j4 + 3] = b.w;
  }
  const int c0 = h * 64 + lane, c1 = c0 + 32;
  const float w0a = vc.w0[c0], w0b = vc.w0[c1], a0a = vc.a0[c0], a0b = vc.a0[c1];
  const float kka = vc.k_k[c0], kkb = vc.k_k[c1], kaa = vc.k_a[c0], kab = vc.k_a[c1];
  const float rka = vc.r_k[c0], rkb = vc.r_k[c1], gwa = vc.gn_w[c0], gwb = vc.gn_w[c1], gba = vc.gn_b[c0], gbb = vc.gn_b[c1];
  float v0a = 0.f, v0b = 0.f;
  if (!LAYER0) {
    v0a = vc.v0[c0];
    v0b = vc.v0[c1];
  }
  // software pipeline: the next row's inputs are loaded while the current row is processed
  float n_r[2], n_k[2], n_v[2], n_wl[2], n_al[2], n_g[2], n_vl[2] = {0.f, 0.f}, n_vf[2] = {0.f, 0.f};
  auto load_row = [&](int row) {
    const size_t b0 = (size_t)row * C + c0, b1 = b0 + 32;
    n_r[0] = io.r[b0]; n_r[1] = io.r[b1];
    n_k[0] = io.k[b0]; n_k[1] = io.k[b1];
    n_v[0] = io.v[b0]; n_v[1] = io.v[b1];
    n_wl[0] = io.wl[b0]; n_wl[1] = io.wl[b1];
    n_al[0] = io.al[b0]; n_al[1] = io.al[b1];
    n_g[0] = io.g[b0]; n_g[1] = io.g[b1];
    if (!LAYER0) {
      n_vl[0] = io.vl[b0]; n_vl[1] = io.vl[b1];
      n_vf[0] = io.v_first[b0]; n_vf[1] = io.v_first[b1];
    }
  };
  load_row(rb);
  for (int row = rb; row < re; row++) {
    const float r0 = n_r[0], r1 = n_r[1], kr0 = n_k[0], kr1 = n_k[1], g0 = n_g[0], g1 = n_g[1];
    float vv0 = n_v[0], vv1 = n_v[1];
    const float wl0 = n_wl[0], wl1 = n_wl[1], al0 = n_al[0], al1 = n_al[1];
    const float vl0 = n_vl[0], vl1 = n_vl[1], vf0 = n_vf[0], vf1 = n_vf[1];
    if (row + 1 < re) load_row(row + 1);
    // decay  w = exp(-exp(-softplus(-(w0 + lora)) - 0.5))   (rwkv7.rs:213-221)
    const float z0 = wl0 + w0a, z1 = wl1 + w0b;
    const float wd0 = expf(-expf(-logf(expf(-z0) + 1.0f) + -0.5f)), wd1 = expf(-expf(-logf(expf(-z1) + 1.0f) + -0.5f));
    const float a0 = sigmoid_f(al0 + a0a), a1 = sigmoid_f(al1 + a0b);  // rwkv7.rs:227-230
    if (LAYER0) {                                                         // rwkv7.rs:238-248
      io.v_first[(size_t)row * C + c0] = vv0;
      io.v_first[(size_t)row * C + c1] = vv1;
    } else {
      vv0 = vv0 + (vf0 - vv0) * sigmoid_f(vl0 + v0a);
      vv1 = vv1 + (vf1 - vv1) * sigmoid_f(vl1 + v0b);
    }
    float kk0 = kr0 * kka, kk1 = kr1 * kkb;  // rwkv7.rs:251-259
    float nrm = sqrtf(warp_sum(fmaf(kk0, kk0, kk1 * kk1)));
    nrm = fmaxf(nrm, 1e-12f);
    kk0 /= nrm;
    kk1 /= nrm;
    const float kp0 = kr0 * (1.0f + (a0 - 1.0f) * kaa), kp1 = kr1 * (1.0f + (a1 - 1.0f) * kab);  // rwkv7.rs:263-265
    __syncwarp();  // previous row's readers are done with the shared vectors
    s_w[lane] = wd0; s_w[lane + 32] = wd1;
    s_kk[lane] = kk0; s_kk[lane + 32] = kk1;
    s_ka[lane] = kk0 * a0; s_ka[lane + 32] = kk1 * a1;
    s_kp[lane] = kp0; s_kp[lane + 32] = kp1;
    s_r[lane] = r0; s_r[lane + 32] = r1;
    __syncwarp();
    // sa = (S kk)[i] with the OLD state (rwkv7.rs:293-295); four partial chains, combined in a fixed order
    float sa0[4] = {0.f, 0.f, 0.f, 0.f}, sa1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j4 = 0; j4 < 16; j4++) {
      const float4 q = *reinterpret_cast<const float4 *>(&s_kk[4 * j4]);
      sa0[0] = fmaf(S0[4 * j4], q.x, sa0[0]); sa0[1] = fmaf(S0[4 * j4 + 1], q.y, sa0[1]);
      sa0[2] = fmaf(S0[4 * j4 + 2], q.z, sa0[2]); sa0[3] = fmaf(S0[4 * j4 + 3], q.w, sa0[3]);
      sa1[0] = fmaf(S1[4 * j4], q.x, sa1[0]); sa1[1] = fmaf(S1[4 * j4 + 1], q.y, sa1[1]);
      sa1[2] = fmaf(S1[4 * j4 + 2], q.z, sa1[2]); sa1[3] = fmaf(S1[4 * j4 + 3], q.w, sa1[3]);
    }
    const float sA = (sa0[0] + sa0[1]) + (sa0[2] + sa0[3]), sB = (sa1[0] + sa1[1]) + (sa1[2] + sa1[3]);
    // S = S*w - sa*(kk*a) + v*k~ ;  y = S r   (rwkv7.rs:290-302)
    float y0[4] = {0.f, 0.f, 0.f, 0.f}, y1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j4 = 0; j4 < 16; j4++) {
      const float4 w4 = *reinterpret_cast<const float4 *>(&s_w[4 * j4]);
      const float4 ka4 = *reinterpret_cast<const float4 *>(&s_ka[4 * j4]);
      const float4 kp4 = *reinterpret_cast<const float4 *>(&s_kp[4 * j4]);
      const float4 r4 = *reinterpret_cast<const float4 *>(&s_r[4 * j4]);
      const float wj[4] = {w4.x, w4.y, w4.z, w4.w}, kaj[4] = {ka4.x, ka4.y, ka4.z, ka4.w};
      const float kpj[4] = {kp4.x, kp4.y, kp4.z, kp4.w}, rj[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int j = 4 * j4 + e;
        S0[j] = fmaf(vv0, kpj[e], fmaf(-sA, kaj[e], S0[j] * wj[e]));
        S1[j] = fmaf(vv1, kpj[e], fmaf(-sB, kaj[e], S1[j] * wj[e]));
        y0[e] = fmaf(S0[j], rj[e], y0[e]);
        y1[e] = fmaf(S1[j], rj[e], y1[e]);
      }
    }
    const float yA = (y0[0] + y0[1]) + (y0[2] + y0[3]), yB = (y1[0] + y1[1]) + (y1[2] + y1[3]);
    // group norm over the head's 64 outputs, eps 64e-5 (rwkv7.rs:312-314, 529-542)
    const float mean = warp_sum(yA + yB) * (1.0f / 64.0f);
    const float dA = yA - mean, dB = yB - mean;
    const float var = warp_sum(fmaf(dA, dA, dB * dB)) * (1.0f / 64.0f);
    const float den = sqrtf(var + 64e-5f);
    // bonus (sum_j r k~ r_k) v   (rwkv7.rs:317-321), gate (324)
    const float alpha = warp_sum(fmaf(r0 * kp0, rka, (r1 * kp1) * rkb));
    const float oA = ((dA / den) * gwa + gba + alpha * vv0) * g0;
    const float oB = ((dB / den) * gwb + gbb + alpha * vv1) * g1;
    out[(size_t)row * C + c0] = __float2bfloat16_rn(oA);
    out[(size_t)row * C + c1] = __float2bfloat16_rn(oB);
  }
#pragma unroll
  for (int j4 = 0; j4 < 16; j4++) {
    st4[j4 * 64 + lane] = make_float4(S0[4 * j4], S0[4 * j4 + 1], S0[4 * j4 + 2], S0[4 * j4 + 3]);
    st4[j4 * 64 + lane + 32] = make_float4(S1[4 * j4], S1[4 * j4 + 1], S1[4 * j4 + 2], S1[4 * j4 + 3]);
  }
}

}  // namespace czk

namespace cz {

// -------------------------------------------------------------------------------------------------------------------------
// weight packing
// -------------------------------------------------------------------------------------------------------------------------
static float bf16_to_f32_host(uint16_t b) {
  uint32_t u = (uint32_t)b << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

int rwkv_finalize(cz_model *m) {
  const cz_model_config &c = m->cfg;
  const size_t C = c.d_model, F = c.d_ffn, L = c.n_layers;
  if (c.head_dim != 64 || C % 64 || C > (size_t)czk::RW_MAXC || F % 64 || c.lora_w % 64 || c.lora_a % 64 || c.lora_g % 64 ||
      c.lora_v <= 0 || c.lora_v > 64) {
    set_error("unsupported RWKV-7 shape (need head_dim 64, d_model % 64 == 0 and <= 1024, d_ffn % 64, LoRA ranks w/a/g % 64, v <= 64)");
    return CZ_ERR_UNSUPPORTED;
  }
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  RwkvWeights &rw = m->rw;
  auto dev = [&](const std::string &name) -> __nv_bfloat16 * { return m->tensors[m->index[name]].dev; };
  // fp32 copies of all vector parameters: [L][RV_COUNT][C] + ln_out (w, b)
  std::vector<float> vecs((L * RV_COUNT + 2) * C, 0.f);
  std::vector<uint16_t> tmp(C);
  auto fetch = [&](const std::string &name, float *dst) -> int {
    CZ_CUDA_TRY(cudaMemcpy(tmp.data(), dev(name), C * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < C; i++) dst[i] = bf16_to_f32_host(tmp[i]);
    return CZ_OK;
  };
  // v-LoRA padded to rank 64 with zeros (K of a tcgen05 GEMM is a multiple of 64; zero rows/columns add exact zeros)
  CZ_CUDA_TRY(cudaMalloc((void **)&rw.v_pad, L * 2 * 64 * C * 2));
  CZ_CUDA_TRY(cudaMemset(rw.v_pad, 0, L * 2 * 64 * C * 2));
  rw.layers.resize(L);
  for (size_t l = 0; l < L; l++) {
    const std::string p = "model.layers." + std::to_string(l) + ".", a = p + "attn.";
    float *v = &vecs[l * RV_COUNT * C];
    if (l == 0) {
      CZ_TRY(fetch(p + "pre_norm.weight", v + RV_PRE_W * C));
      CZ_TRY(fetch(p + "pre_norm.bias", v + RV_PRE_B * C));
    }
    CZ_TRY(fetch(p + "attn_norm.weight", v + RV_LN1_W * C));
    CZ_TRY(fetch(p + "attn_norm.bias", v + RV_LN1_B * C));
    CZ_TRY(fetch(p + "ffn_norm.weight", v + RV_LN2_W * C));
    CZ_TRY(fetch(p + "ffn_norm.bias", v + RV_LN2_B * C));
    const char *mixn[6] = {"x_r", "x_w", "x_k", "x_v", "x_a", "x_g"};
    for (int q = 0; q < 6; q++) CZ_TRY(fetch(a + mixn[q], v + (RV_XR + q) * C));
    CZ_TRY(fetch(a + "k_k", v + RV_KK * C));
    CZ_TRY(fetch(a + "k_a", v + RV_KA * C));
    CZ_TRY(fetch(a + "r_k", v + RV_RK * C));
    CZ_TRY(fetch(a + "w_lora.lora.2.bias", v + RV_W0 * C));
    CZ_TRY(fetch(a + "a_lora.lora.2.bias", v + RV_A0 * C));
    if (l > 0) CZ_TRY(fetch(a + "v_lora.lora.2.bias", v + RV_V0 * C));
    CZ_TRY(fetch(a + "g_norm.weight", v + RV_GNW * C));
    CZ_TRY(fetch(a + "g_norm.bias", v + RV_GNB * C));
    CZ_TRY(fetch(p + "ffn.x_k", v + RV_FXK * C));
    RwkvLayerW &W = rw.layers[l];
    W.wr = dev(a + "r_proj.weight");
    W.wk = dev(a + "k_proj.weight");
    W.wv = dev(a + "v_proj.weight");
    W.wo = dev(a + "o_proj.weight");
    W.w1 = dev(a + "w_lora.lora.0.weight");
    W.w2 = dev(a + "w_lora.lora.2.weight");
    W.a1 = dev(a + "a_lora.lora.0.weight");
    W.a2 = dev(a + "a_lora.lora.2.weight");
    W.g1 = dev(a + "g_lora.lora.0.weight");
    W.g2 = dev(a + "g_lora.lora.2.weight");
    W.fk = dev(p + "ffn.key.weight");
    W.fv = dev(p + "ffn.value.weight");
    W.v1 = W.v2 = nullptr;
    if (l > 0) {
      W.v1 = rw.v_pad + (l * 2) * 64 * C;      // [64][C], rows >= lora_v zero
      W.v2 = rw.v_pad + (l * 2 + 1) * 64 * C;  // [C][64], columns >= lora_v zero
      CZ_CUDA_TRY(cudaMemcpy(W.v1, dev(a + "v_lora.lora.0.weight"), (size_t)c.lora_v * C * 2, cudaMemcpyDeviceToDevice));
      CZ_CUDA_TRY(cudaMemcpy2D(W.v2, 64 * 2, dev(a + "v_lora.lora.2.weight"), (size_t)c.lora_v * 2, (size_t)c.lora_v * 2, C,
                               cudaMemcpyDeviceToDevice));
    }
  }
  CZ_TRY(fetch("model.norm.weight", &vecs[L * RV_COUNT * C]));
  CZ_TRY(fetch("model.norm.bias", &vecs[(L * RV_COUNT + 1) * C]));
  CZ_CUDA_TRY(cudaMalloc((void **)&rw.vecs, vecs.size() * 4));
  CZ_CUDA_TRY(cudaMemcpy(rw.vecs, vecs.data(), vecs.size() * 4, cudaMemcpyHostToDevice));
  m->embed = dev("model.embeddings.weight");
  m->head_w = dev("lm_head.weight");
  return CZ_OK;
}

template <typename T>
static int rw_realloc(T *&p, size_t n) {
  if (p) cudaFree(p);
  p = nullptr;
  if (n == 0) return CZ_OK;
  CZ_CUDA_TRY(cudaMalloc((void **)&p, n * sizeof(T)));
  return CZ_OK;
}

int rwkv_ensure_ws(cz_model *m, size_t rows, size_t n_streams) {
  RwkvWs &w = m->rws;
  const cz_model_config &c = m->cfg;
  const size_t C = c.d_model, F = c.d_ffn;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (rows > w.cap_rows) {
    CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
    const size_t r = rows + rows / 8 + 128;
    for (int q = 0; q < 6; q++) CZ_TRY(rw_realloc(w.mix[q], r * C));
    for (int q = 0; q < 7; q++) CZ_TRY(rw_realloc(w.f[q], r * C));
    CZ_TRY(rw_realloc(w.v_first, r * C));
    CZ_TRY(rw_realloc(w.lo, r * 128));
    CZ_TRY(rw_realloc(w.att, r * C));
    CZ_TRY(rw_realloc(w.act, r * F));
    CZ_TRY(rw_realloc(w.prev_row, r));
    CZ_TRY(rw_realloc(w.slot, r));
    CZ_TRY(rw_realloc(w.flags, r));
    w.cap_rows = r;
  }
  if (n_streams > w.cap_streams) {
    CZ_CUDA_TRY(cudaStreamSynchronize(m->ctx->stream));
    const size_t s = n_streams + n_streams / 8 + 16;
    CZ_TRY(rw_realloc(w.row_begin, s));
    CZ_TRY(rw_realloc(w.row_end, s));
    CZ_TRY(rw_realloc(w.stream_slot, s));
    w.cap_streams = s;
  }
  return CZ_OK;
}

// state for `n` stream slots, zero-initialised (State::new, rwkv7.rs:47-60)
int rwkv_state_reset(cz_model *m, RwkvState &s, size_t n, cudaStream_t st) {
  const cz_model_config &c = m->cfg;
  const size_t C = c.d_model, L = c.n_layers, H = C / 64;
  CZ_CUDA_TRY(cudaSetDevice(m->ctx->device));
  if (n > s.cap) {
    CZ_CUDA_TRY(cudaStreamSynchronize(st));
    CZ_TRY(rw_realloc(s.S, L * n * H * 4096));
    for (int p = 0; p < 2; p++) {
      CZ_TRY(rw_realloc(s.xa[p], L * n * C));
      CZ_TRY(rw_realloc(s.xf[p], L * n * C));
    }
    s.cap = n;
  }
  s.n = n;
  s.cur = 0;
  CZ_CUDA_TRY(cudaMemsetAsync(s.S, 0, L * s.cap * H * 4096 * 4, st));
  for (int p = 0; p < 2; p++) {
    CZ_CUDA_TRY(cudaMemsetAsync(s.xa[p], 0, L * s.cap * C * 4, st));
    CZ_CUDA_TRY(cudaMemsetAsync(s.xf[p], 0, L * s.cap * C * 4, st));
  }
  return CZ_OK;
}

void rwkv_state_free(RwkvState &s) {
  if (s.S) cudaFree(s.S);
  for (int p = 0; p < 2; p++) {
    if (s.xa[p]) cudaFree(s.xa[p]);
    if (s.xf[p]) cudaFree(s.xf[p]);
  }
  s = RwkvState();
}

void rwkv_free(cz_model *m) {
  RwkvWs &w = m->rws;
  void *ptrs[] = {w.mix[0], w.mix[1], w.mix[2], w.mix[3], w.mix[4], w.mix[5], w.f[0], w.f[1], w.f[2], w.f[3], w.f[4], w.f[5], w.f[6],
                  w.v_first, w.lo, w.att, w.act, w.prev_row, w.slot, w.flags, w.row_begin, w.row_end, w.stream_slot, m->rw.v_pad,
                  m->rw.vecs};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  rwkv_state_free(m->rstate);
}

// Forward of one slab.  Row metadata (ws.tok; rws.prev_row/slot/flags; rws.row_begin/row_end/stream_slot) is already on the
// device.  in_place: T = 1 decode steps read and write the same token-shift buffers; slabs ping-pong them.
// stream_active (device, nullable): per-stream flag for the stepwise decoder.

// rwkv_ln_mix takes the 8-elements-per-lane kernel when the width is a multiple of 256 (<= 1024) and every operand is 16-byte aligned
template <int NMIX>
static bool ln_mix_takes_v8(int C, const float *x, const float *lnw, const float *lnb, const czk::MixMu &mu, const float *state_in,
                            const float *state_out, const czk::MixOut &out) {
  bool vec = C % 256 == 0 && C <= 1024 && (((uintptr_t)x | (uintptr_t)lnw | (uintptr_t)lnb | (uintptr_t)state_in | (uintptr_t)state_out) & 15) == 0;
  for (int q = 0; q < NMIX; q++) vec = vec && (((uintptr_t)mu.p[q] | (uintptr_t)out.p[q]) & 15) == 0;
  return vec;
}

// lane_form: run the element-per-lane kernel even where the v8 form applies (cz_test_rwkv_ln_mix compares the two)
template <int NMIX>
static int launch_ln_mix(cz_ctx *ctx, cudaStream_t st, unsigned grid, const float *x, const float *lnw, const float *lnb, const czk::MixMu &mu,
                         const int *prev_row, const int *slot, const int *flags, const float *state_in, float *state_out, const czk::MixOut &out,
                         int n_rows, int C, float eps, bool lane_form = false) {
  const bool vec = !lane_form && ln_mix_takes_v8<NMIX>(C, x, lnw, lnb, mu, state_in, state_out, out);
#define CZ_LNMIX_V8(NCH)                                                                                                                       \
  CZ_LAUNCH(ctx, CZ_K_ELEMWISE,                                                                                                                \
            (czk::rwkv_ln_mix_v8_kernel<NMIX, NCH><<<grid, 128, 0, st>>>(x, lnw, lnb, mu, prev_row, slot, flags, state_in, state_out, out, n_rows, \
                                                                        eps)))
  if (vec && C == 256) CZ_LNMIX_V8(1);
  else if (vec && C == 512) CZ_LNMIX_V8(2);
  else if (vec && C == 768) CZ_LNMIX_V8(3);
  else if (vec && C == 1024) CZ_LNMIX_V8(4);
  else
    CZ_LAUNCH(ctx, CZ_K_ELEMWISE,
              (czk::rwkv_ln_mix_kernel<NMIX><<<grid, 128, 0, st>>>(x, lnw, lnb, mu, prev_row, slot, flags, state_in, state_out, out, n_rows, C, eps)));
#undef CZ_LNMIX_V8
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

// one WKV-7 scan: a warp per (stream, head); S is one layer's state [n_slots][H][4096]
static int launch_wkv7_scan(cz_ctx *ctx, cudaStream_t st, bool layer0, const czk::WkvIo &io, const czk::WkvVecs &vc, const int *row_begin,
                            const int *row_end, const int *stream_slot, const int *stream_active, float *S, __nv_bfloat16 *out, int n_streams,
                            int C) {
  const int H = C / 64;
  const dim3 grid((unsigned)n_streams, (unsigned)H);
  if (layer0)
    CZ_LAUNCH(ctx, CZ_K_ATTN, (czk::wkv7_scan_kernel<true><<<grid, 32, 0, st>>>(io, vc, row_begin, row_end, stream_slot, stream_active, S, out, C, H)));
  else
    CZ_LAUNCH(ctx, CZ_K_ATTN, (czk::wkv7_scan_kernel<false><<<grid, 32, 0, st>>>(io, vc, row_begin, row_end, stream_slot, stream_active, S, out, C, H)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

int rwkv_forward(cz_model *m, int n_rows, int n_streams, RwkvState &stt, bool in_place, const int *stream_active, cudaStream_t st) {
  const cz_model_config &c = m->cfg;
  cz_ctx *ctx = m->ctx;
  Workspace &ws = m->ws;
  RwkvWs &w = m->rws;
  const int C = c.d_model, F = c.d_ffn, L = c.n_layers, H = C / 64;
  const size_t cap = stt.cap;
  const int pin = stt.cur, pout = in_place ? stt.cur : stt.cur ^ 1;
  const unsigned g4 = (unsigned)ceil_div(n_rows, 4);
  CZ_TRY(launch_embed(ctx, m->embed, ws.tok, ws.x, n_rows, C, c.vocab, st));
  for (int l = 0; l < L; l++) {
    const float *v = m->rw.vecs + (size_t)l * RV_COUNT * C;
    const RwkvLayerW &W = m->rw.layers[l];
    if (l == 0) {
      CZ_LAUNCH(ctx, CZ_K_ELEMWISE,
                (czk::rwkv_ln_inplace_kernel<<<g4, 128, 0, st>>>(ws.x, v + RV_PRE_W * C, v + RV_PRE_B * C, n_rows, C, c.norm_eps)));
      CZ_CHECK_LAUNCH();
    }
    czk::MixMu mu{};
    czk::MixOut mo{};
    for (int q = 0; q < 6; q++) {
      mu.p[q] = v + (size_t)(RV_XR + q) * C;
      mo.p[q] = w.mix[q];
    }
    CZ_TRY(launch_ln_mix<6>(ctx, st, g4, ws.x, v + RV_LN1_W * C, v + RV_LN1_B * C, mu, w.prev_row, w.slot, w.flags,
                            stt.xa[pin] + (size_t)l * cap * C, stt.xa[pout] + (size_t)l * cap * C, mo, n_rows, C, c.norm_eps));
    // f[0]=r f[1]=k f[2]=v f[3]=w-lora f[4]=a-lora f[5]=v-lora f[6]=g
    auto mm = [&](const __nv_bfloat16 *a, int lda, const __nv_bfloat16 *b, int K, int N, void *out, int ldc, int epi, int bn, int fam) {
      GemmArgs g{};
      g.a = a; g.lda = lda; g.b = b; g.ldb = K; g.c = out; g.ldc = ldc; g.M = n_rows; g.N = N; g.K = K; g.epi = epi; g.bn = bn; g.fam = fam;
      return gemm(ctx, c.engine, g, st);
    };
    CZ_TRY(mm(w.mix[0], C, W.wr, C, C, w.f[0], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.mix[2], C, W.wk, C, C, w.f[1], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.mix[3], C, W.wv, C, C, w.f[2], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.mix[1], C, W.w1, C, c.lora_w, w.lo, 128, EPI_TANH_BF16, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.lo, 128, W.w2, c.lora_w, C, w.f[3], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.mix[4], C, W.a1, C, c.lora_a, w.lo, 128, EPI_STORE_BF16, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.lo, 128, W.a2, c.lora_a, C, w.f[4], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    if (l > 0) {
      CZ_TRY(mm(w.mix[3], C, W.v1, C, 64, w.lo, 128, EPI_STORE_BF16, 192, CZ_K_GEMM));
      CZ_TRY(mm(w.lo, 128, W.v2, 64, C, w.f[5], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    }
    CZ_TRY(mm(w.mix[5], C, W.g1, C, c.lora_g, w.lo, 128, EPI_SIGMOID_BF16, 192, CZ_K_GEMM));
    CZ_TRY(mm(w.lo, 128, W.g2, c.lora_g, C, w.f[6], C, EPI_STORE_F32, 192, CZ_K_GEMM));
    czk::WkvIo io{w.f[0], w.f[1], w.f[2], w.f[3], w.f[4], w.f[5], w.f[6], w.v_first};
    czk::WkvVecs vc{v + RV_W0 * C, v + RV_A0 * C, v + RV_V0 * C, v + RV_KK * C, v + RV_KA * C, v + RV_RK * C, v + RV_GNW * C, v + RV_GNB * C};
    CZ_TRY(launch_wkv7_scan(ctx, st, l == 0, io, vc, w.row_begin, w.row_end, w.stream_slot, stream_active, stt.S + (size_t)l * cap * H * 4096,
                            w.att, n_streams, C));
    CZ_TRY(mm(w.att, C, W.wo, C, C, ws.x, C, EPI_ADD_F32, 192, CZ_K_GEMM_O));
    // feed-forward
    czk::MixMu mu1{};
    czk::MixOut mo1{};
    mu1.p[0] = v + (size_t)RV_FXK * C;
    mo1.p[0] = w.mix[0];
    CZ_TRY(launch_ln_mix<1>(ctx, st, g4, ws.x, v + RV_LN2_W * C, v + RV_LN2_B * C, mu1, w.prev_row, w.slot, w.flags,
                            stt.xf[pin] + (size_t)l * cap * C, stt.xf[pout] + (size_t)l * cap * C, mo1, n_rows, C, c.norm_eps));
    CZ_TRY(mm(w.mix[0], C, W.fk, C, F, w.act, F, EPI_RELUSQ_BF16, 256, CZ_K_GEMM_GU));
    CZ_TRY(mm(w.act, F, W.fv, F, C, ws.x, C, EPI_ADD_F32, 192, CZ_K_GEMM_DOWN));
  }
  if (!in_place) stt.cur ^= 1;
  return CZ_OK;
}

// final LayerNorm of the rows listed in ws.logit_rows -> ws.xn_logit
int rwkv_final_norm_gather(cz_model *m, int n_logit, cudaStream_t st) {
  const cz_model_config &c = m->cfg;
  const int C = c.d_model;
  const float *v = m->rw.vecs + (size_t)c.n_layers * RV_COUNT * C;
  if (n_logit == 0) return CZ_OK;
  CZ_LAUNCH(m->ctx, CZ_K_ELEMWISE,
            (czk::rwkv_ln_gather_kernel<<<(unsigned)ceil_div(n_logit, 4), 128, 0, st>>>(m->ws.x, v, v + C, m->ws.logit_rows, m->ws.xn_logit,
                                                                                       n_logit, C, c.norm_eps)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

}  // namespace cz

// ---- test hooks (declared in include/candlezip_b200.h): the two RWKV-7 kernel families on host buffers, through the launchers
// rwkv_forward uses, so tests can compare them with an f64 restatement at shapes and edges the model never produces on its own
namespace cz {
int require_device(cz_ctx *ctx);

namespace {
struct HookBufs {  // the device buffers of one hook call, freed on every return path
  std::vector<void *> p;
  ~HookBufs() {
    for (void *q : p) cudaFree(q);
  }
  template <typename T>
  int alloc(T *&out, size_t n) {
    void *q = nullptr;
    CZ_CUDA_TRY(cudaMalloc(&q, std::max<size_t>(n * sizeof(T), 16)));
    p.push_back(q);
    out = (T *)q;
    return CZ_OK;
  }
};

int hook_sync(cz_ctx *ctx, int rc, const char *what) {
  if (rc != CZ_OK) return rc;
  const cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) {
    set_error(std::string(what) + " execution failed: " + cudaGetErrorString(e));
    return CZ_ERR_CUDA;
  }
  return CZ_OK;
}

template <int NMIX>
int hook_ln_mix(cz_ctx *ctx, bool lane_form, int R, int C, const float *x, const float *lnw, const float *lnb, const float *mu,
                const int *meta, const float *state_in, float *state_out, __nv_bfloat16 *out, float eps, int *form_used) {
  czk::MixMu m{};
  czk::MixOut o{};
  for (int q = 0; q < NMIX; q++) {
    m.p[q] = mu + (size_t)q * C;
    o.p[q] = out + (size_t)q * R * C;
  }
  *form_used = !lane_form && ln_mix_takes_v8<NMIX>(C, x, lnw, lnb, m, state_in, state_out, o) ? 8 : 1;
  return launch_ln_mix<NMIX>(ctx, ctx->stream, (unsigned)ceil_div(R, 4), x, lnw, lnb, m, meta, meta + R, meta + 2 * R, state_in, state_out, o, R,
                             C, eps, lane_form);
}
}  // namespace
}  // namespace cz

extern "C" int cz_test_wkv7_scan(cz_ctx *ctx, int layer0, int R, int H, int n_streams, const int *row_begin, const int *row_end,
                                 const int *stream_slot, const int *stream_active, int n_slots, const float *rows, float *v_first,
                                 const float *vecs, float *state, uint16_t *out_bf16) {
  using namespace cz;
  CZ_TRY(require_device(ctx));
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  bool ok = R > 0 && H >= 1 && H <= czk::RW_MAXC / 64 && n_streams > 0 && n_slots > 0 && row_begin && row_end && stream_slot && rows &&
            v_first && vecs && state && out_bf16;
  for (int s = 0; ok && s < n_streams; s++)
    ok = row_begin[s] >= 0 && row_end[s] <= R && stream_slot[s] >= 0 && stream_slot[s] < n_slots;
  if (!ok) {
    set_error("cz_test_wkv7_scan: bad arguments");
    return CZ_ERR_INVALID;
  }
  const int C = 64 * H;
  const size_t RC = (size_t)R * C, SN = (size_t)n_slots * H * 4096, NS = (size_t)n_streams;
  HookBufs d;
  float *drows, *dvf, *dvecs, *dS;
  __nv_bfloat16 *dout;
  int *dmeta;
  CZ_TRY(d.alloc(drows, 7 * RC));
  CZ_TRY(d.alloc(dvf, RC));
  CZ_TRY(d.alloc(dvecs, 8 * (size_t)C));
  CZ_TRY(d.alloc(dS, SN));
  CZ_TRY(d.alloc(dout, RC));
  CZ_TRY(d.alloc(dmeta, 4 * NS));
  CZ_CUDA_TRY(cudaMemcpy(drows, rows, 7 * RC * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dvf, v_first, RC * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dvecs, vecs, 8 * (size_t)C * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dS, state, SN * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dout, out_bf16, RC * 2, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmeta, row_begin, NS * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmeta + NS, row_end, NS * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmeta + 2 * NS, stream_slot, NS * 4, cudaMemcpyHostToDevice));
  if (stream_active) CZ_CUDA_TRY(cudaMemcpy(dmeta + 3 * NS, stream_active, NS * 4, cudaMemcpyHostToDevice));
  const czk::WkvIo io{drows, drows + RC, drows + 2 * RC, drows + 3 * RC, drows + 4 * RC, drows + 5 * RC, drows + 6 * RC, dvf};
  const czk::WkvVecs vc{dvecs, dvecs + C, dvecs + 2 * C, dvecs + 3 * C, dvecs + 4 * C, dvecs + 5 * C, dvecs + 6 * C, dvecs + 7 * C};
  CZ_TRY(hook_sync(ctx,
                   launch_wkv7_scan(ctx, ctx->stream, layer0 != 0, io, vc, dmeta, dmeta + NS, dmeta + 2 * NS, stream_active ? dmeta + 3 * NS : nullptr,
                                    dS, dout, n_streams, C),
                   "wkv7 scan"));
  CZ_CUDA_TRY(cudaMemcpy(v_first, dvf, RC * 4, cudaMemcpyDeviceToHost));
  CZ_CUDA_TRY(cudaMemcpy(state, dS, SN * 4, cudaMemcpyDeviceToHost));
  CZ_CUDA_TRY(cudaMemcpy(out_bf16, dout, RC * 2, cudaMemcpyDeviceToHost));
  return CZ_OK;
}

extern "C" int cz_test_rwkv_ln_mix(cz_ctx *ctx, int nmix, int form, int in_place, int R, int C, int n_slots, const float *x, const float *lnw,
                                   const float *lnb, const float *mu, const int *prev_row, const int *slot, const int *flags,
                                   const float *state_in, float *state_out, float eps, uint16_t *out_bf16, int *form_used) {
  using namespace cz;
  CZ_TRY(require_device(ctx));
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  bool ok = (nmix == 1 || nmix == 6) && (form == 0 || form == 1) && R > 0 && C > 0 && C <= czk::RW_MAXC && n_slots > 0 && x && lnw && lnb &&
            mu && prev_row && slot && flags && state_in && state_out && out_bf16 && form_used;
  for (int r = 0; ok && r < R; r++) ok = prev_row[r] >= -1 && prev_row[r] < R && slot[r] >= 0 && slot[r] < n_slots;
  if (!ok) {
    set_error("cz_test_rwkv_ln_mix: bad arguments");
    return CZ_ERR_INVALID;
  }
  const size_t RC = (size_t)R * C, SN = (size_t)n_slots * C;
  HookBufs d;
  float *dx, *dw, *db, *dmu, *dsin, *dsout;
  __nv_bfloat16 *dout;
  int *dmeta;
  CZ_TRY(d.alloc(dx, RC));
  CZ_TRY(d.alloc(dw, (size_t)C));
  CZ_TRY(d.alloc(db, (size_t)C));
  CZ_TRY(d.alloc(dmu, (size_t)nmix * C));
  CZ_TRY(d.alloc(dsin, SN));
  CZ_TRY(d.alloc(dout, (size_t)nmix * RC));
  CZ_TRY(d.alloc(dmeta, 3 * (size_t)R));
  if (in_place) {
    dsout = dsin;  // the stepwise decoder's T = 1 steps read and write the same token-shift rows
  } else {
    CZ_TRY(d.alloc(dsout, SN));
    CZ_CUDA_TRY(cudaMemcpy(dsout, state_out, SN * 4, cudaMemcpyHostToDevice));
  }
  CZ_CUDA_TRY(cudaMemcpy(dx, x, RC * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dw, lnw, (size_t)C * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(db, lnb, (size_t)C * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmu, mu, (size_t)nmix * C * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dsin, state_in, SN * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemset(dout, 0xff, (size_t)nmix * RC * 2));  // NaN: a row the kernel skips cannot pass for a result
  CZ_CUDA_TRY(cudaMemcpy(dmeta, prev_row, (size_t)R * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmeta + R, slot, (size_t)R * 4, cudaMemcpyHostToDevice));
  CZ_CUDA_TRY(cudaMemcpy(dmeta + 2 * R, flags, (size_t)R * 4, cudaMemcpyHostToDevice));
  const bool lane = form == 1;
  const int rc = nmix == 6 ? hook_ln_mix<6>(ctx, lane, R, C, dx, dw, db, dmu, dmeta, dsin, dsout, dout, eps, form_used)
                           : hook_ln_mix<1>(ctx, lane, R, C, dx, dw, db, dmu, dmeta, dsin, dsout, dout, eps, form_used);
  CZ_TRY(hook_sync(ctx, rc, "rwkv ln-mix"));
  CZ_CUDA_TRY(cudaMemcpy(state_out, dsout, SN * 4, cudaMemcpyDeviceToHost));
  CZ_CUDA_TRY(cudaMemcpy(out_bf16, dout, (size_t)nmix * RC * 2, cudaMemcpyDeviceToHost));
  return CZ_OK;
}
