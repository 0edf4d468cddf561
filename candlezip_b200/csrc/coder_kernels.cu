// K2 / K3 lane kernels: one thread per independent arithmetic-coder stream (segment).
// Replaces ArithmeticEncoder::{encode_counts, finish} (src/main.rs:353-399) and
// ArithmeticDecoder::{new, decode_symbol_counts} (src/main.rs:419-437, 500-548).
// Bytes are negligible (8 B in, <= 4 B out per symbol); what matters is that every lane advances
// independently and the output is bit-identical to the reference's single-threaded coder.
#include "coder.cuh"
#include "cz_common.cuh"

namespace czk {

// One WARP per lane: the 32 threads prefetch the next AC_BATCH intervals into shared memory with coalesced loads and
// flush the produced bytes with coalesced stores; thread 0 runs the (inherently sequential) coder out of shared memory.
// A single thread reading (c_lo, c_hi) straight from global memory pays a full DRAM round trip per symbol.
// err[0]: OR of status bits; err_index: smallest interval index that had zero width (atomicMin).
// LANE_ZW (cz_model_set_zero_width_out): every lane also writes lane_zw[lane], the lane-relative index of its own first zero-width
// interval or ~0 when it has none, so that one segment's zero-width token does not make the caller re-code the other segments.
constexpr int AC_BATCH = 512;
constexpr int AC_STAGE = 4096;
template <bool LANE_ZW>
__global__ void __launch_bounds__(32) ac_encode_lanes_kernel(const uint32_t *__restrict__ c_lo, const uint32_t *__restrict__ c_hi,
                                                             const uint64_t *__restrict__ lane_off, size_t n_lanes,
                                                             uint8_t *__restrict__ out, const uint64_t *__restrict__ out_off,
                                                             uint64_t *__restrict__ out_len, int *__restrict__ err,
                                                             unsigned long long *__restrict__ err_index,
                                                             unsigned long long *__restrict__ lane_zw) {
  __shared__ uint32_t s_lo[AC_BATCH], s_hi[AC_BATCH];
  __shared__ __align__(16) uint8_t s_stage[AC_STAGE];
  const size_t lane = blockIdx.x;
  if (lane >= n_lanes) return;
  const int tid = threadIdx.x;
  AcEncoder enc;
  enc.init(out + out_off[lane]);
  enc.stage = s_stage;
  enc.stage_cap = AC_STAGE;
  const uint64_t t0 = lane_off[lane], t1 = lane_off[lane + 1];
  uint8_t *gout = out + out_off[lane];
  for (uint64_t base = t0; base < t1; base += AC_BATCH) {
    const int cnt = (int)((t1 - base) < (uint64_t)AC_BATCH ? (t1 - base) : (uint64_t)AC_BATCH);
    for (int i = tid; i < cnt; i += 32) {
      s_lo[i] = __ldg(c_lo + base + i);
      s_hi[i] = __ldg(c_hi + base + i);
    }
    __syncwarp();
    int bad = 0;
    if (tid == 0) {
      for (int i = 0; i < cnt; i++) {
        const uint32_t lo = s_lo[i], hi = s_hi[i];
        if (hi <= lo || hi > CZ_AC_CDF_TOTAL) {
          atomicOr(err, 4);
          atomicMin(err_index, (unsigned long long)(base + i));
          if constexpr (LANE_ZW) lane_zw[lane] = (unsigned long long)(base + i - t0);
          bad = 1;
          break;
        }
        enc.encode_counts(lo, hi);
      }
    }
    bad = __shfl_sync(0xffffffffu, bad, 0);
    if (bad) {
      if (tid == 0) out_len[lane] = 0;
      return;
    }
    // cooperative flush of the staged bytes
    __syncwarp();  // thread 0's shared-memory writes -> visible to the warp
    const uint32_t n_st = __shfl_sync(0xffffffffu, enc.stage_n, 0);
    const uint64_t b0 = __shfl_sync(0xffffffffu, (unsigned long long)(enc.n_bytes - enc.stage_n), 0);
    for (uint32_t i = tid; i < n_st; i += 32) gout[b0 + i] = s_stage[i];
    __syncwarp();
    if (tid == 0) enc.stage_n = 0;
  }
  if (tid == 0) {
    const uint64_t total = enc.finish();
    enc.flush_stage_serial();
    out_len[lane] = total;
    if constexpr (LANE_ZW) lane_zw[lane] = ~0ull;
  }
}

__global__ void ac_decode_lanes_static_kernel(const uint8_t *__restrict__ payload, const uint64_t *__restrict__ pay_off,
                                              const uint64_t *__restrict__ pay_len, const uint64_t *__restrict__ lane_off,
                                              size_t n_lanes, const uint32_t *__restrict__ cdf, uint32_t n_sym,
                                              uint32_t *__restrict__ syms_out) {
  size_t lane = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (lane >= n_lanes) return;
  AcDecoder dec;
  dec.init(payload + pay_off[lane], pay_len[lane]);
  for (uint64_t t = lane_off[lane]; t < lane_off[lane + 1]; t++) {
    const uint32_t value = dec.peek_value();
    // same binary search as src/main.rs:508-513
    uint32_t lo = 0, hi = n_sym;
    while (lo + 1 < hi) {
      uint32_t mid = (lo + hi) >> 1;
      if (__ldg(cdf + mid) <= value) lo = mid;
      else hi = mid;
    }
    dec.consume(__ldg(cdf + lo), __ldg(cdf + lo + 1));
    syms_out[t] = lo;
  }
}

}  // namespace czk

namespace cz {

int launch_ac_encode_lanes(cz_ctx *ctx, const uint32_t *c_lo_dev, const uint32_t *c_hi_dev, const uint64_t *lane_off_dev,
                           size_t n_lanes, uint8_t *out_dev, const uint64_t *out_off_dev, uint64_t *out_len_dev,
                           unsigned long long *err_index_dev, cudaStream_t stream, unsigned long long *lane_zw_dev) {
  if (n_lanes == 0) return CZ_OK;
  if (lane_zw_dev)
    CZ_LAUNCH(ctx, CZ_K_CODER,
              (czk::ac_encode_lanes_kernel<true><<<(unsigned)n_lanes, 32, 0, stream>>>(
                  c_lo_dev, c_hi_dev, lane_off_dev, n_lanes, out_dev, out_off_dev, out_len_dev, ctx->err_flag_dev,
                  err_index_dev, lane_zw_dev)));
  else
    CZ_LAUNCH(ctx, CZ_K_CODER,
              (czk::ac_encode_lanes_kernel<false><<<(unsigned)n_lanes, 32, 0, stream>>>(
                  c_lo_dev, c_hi_dev, lane_off_dev, n_lanes, out_dev, out_off_dev, out_len_dev, ctx->err_flag_dev,
                  err_index_dev, nullptr)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

int launch_ac_decode_lanes_static(cz_ctx *ctx, const uint8_t *payload_dev, const uint64_t *pay_off_dev,
                                  const uint64_t *pay_len_dev, const uint64_t *lane_off_dev, size_t n_lanes,
                                  const uint32_t *cdf_dev, uint32_t n_sym, uint32_t *syms_dev, cudaStream_t stream) {
  if (n_lanes == 0) return CZ_OK;
  const int threads = 32;
  CZ_LAUNCH(ctx, CZ_K_CODER,
            (czk::ac_decode_lanes_static_kernel<<<(unsigned)ceil_div(n_lanes, threads), threads, 0, stream>>>(
                payload_dev, pay_off_dev, pay_len_dev, lane_off_dev, n_lanes, cdf_dev, n_sym, syms_dev)));
  CZ_CHECK_LAUNCH();
  return CZ_OK;
}

}  // namespace cz
