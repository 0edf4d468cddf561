// C-ABI: context, error reporting, and the host-buffer entry points of K1 (CDF) and K2/K3 (coder lanes).
// See include/candlezip_b200.h for the reference interfaces each entry point replaces.
#include <string.h>

#include <vector>

#include "cz_common.cuh"

namespace cz {

static thread_local std::string g_err;
void set_error(const std::string &msg) { g_err = msg; }
const char *get_error() { return g_err.c_str(); }

int ensure_scratch(cz_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->scratch_bytes) return CZ_OK;
  if (ctx->scratch) cudaFree(ctx->scratch);
  ctx->scratch = nullptr;
  ctx->scratch_bytes = 0;
  size_t want = bytes + (bytes >> 2) + 4096;
  CZ_CUDA_TRY(cudaMalloc(&ctx->scratch, want));
  ctx->scratch_bytes = want;
  return CZ_OK;
}

// declared in the kernel translation units
int launch_cdf_cols(cz_ctx *ctx, int op, int mode, const float *logits_dev, size_t V, size_t M, size_t ld,
                    const uint32_t *arg_dev, uint32_t *sym_out_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev,
                    double *xe_dev, cudaStream_t stream, const int *colmax_dev = nullptr);
int launch_cdf_full(cz_ctx *ctx, int mode, const float *logits_dev, size_t V, uint32_t *cdf_dev, cudaStream_t stream);
int launch_ac_encode_lanes(cz_ctx *ctx, const uint32_t *c_lo_dev, const uint32_t *c_hi_dev, const uint64_t *lane_off_dev,
                           size_t n_lanes, uint8_t *out_dev, const uint64_t *out_off_dev, uint64_t *out_len_dev,
                           unsigned long long *err_index_dev, cudaStream_t stream, unsigned long long *lane_zw_dev = nullptr);
int launch_ac_decode_lanes_static(cz_ctx *ctx, const uint8_t *payload_dev, const uint64_t *pay_off_dev,
                                  const uint64_t *pay_len_dev, const uint64_t *lane_off_dev, size_t n_lanes,
                                  const uint32_t *cdf_dev, uint32_t n_sym, uint32_t *syms_dev, cudaStream_t stream);

int require_device(cz_ctx *ctx) {
  if (!ctx) {
    set_error("null ctx");
    return CZ_ERR_INVALID;
  }
  if (ctx->device < 0) {
    set_error("this ctx has no GPU (opened with device_id=-1); compute entry points need an sm_100 device");
    return CZ_ERR_NO_DEVICE;
  }
  return CZ_OK;
}

// reads and clears the device status word; maps it to a cz_status.  ignore_bits: status bits the caller reports some other way
// (the zero-width bit when a per-segment zero-width sink is set)
int fetch_device_status_masked(cz_ctx *ctx, unsigned long long *err_index_dev, unsigned long long *err_index_out, int ignore_bits) {
  int flag = 0;
  CZ_CUDA_TRY(cudaMemcpyAsync(&flag, ctx->err_flag_dev, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  unsigned long long idx = ~0ull;
  if (err_index_dev)
    CZ_CUDA_TRY(cudaMemcpyAsync(&idx, err_index_dev, sizeof(idx), cudaMemcpyDeviceToHost, ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (flag) CZ_CUDA_TRY(cudaMemsetAsync(ctx->err_flag_dev, 0, sizeof(int), ctx->stream));
  if (err_index_out) *err_index_out = idx;
  flag &= ~ignore_bits;
  if (flag & 2) {  // (checked before the zero-width bit: an out-of-range symbol also yields an empty interval)
    set_error("symbol id out of range for the coded alphabet");
    return CZ_ERR_SYMBOL_RANGE;
  }
  if (flag & 4) {
    set_error("zero-width coding interval (c_lo == c_hi) at coded index " + std::to_string(idx) +
              ": symbol mass < 2^-30; the reference would corrupt the stream here");
    return CZ_ERR_ZERO_WIDTH;
  }
  if (flag & 1) {
    set_error("NaN in logits");
    return CZ_ERR_INVALID;
  }
  return CZ_OK;
}
int fetch_device_status(cz_ctx *ctx, unsigned long long *err_index_dev, unsigned long long *err_index_out) {
  return fetch_device_status_masked(ctx, err_index_dev, err_index_out, 0);
}

}  // namespace cz

using namespace cz;

extern "C" {

int cz_abi_version(void) { return CZ_ABI_VERSION; }
const char *cz_last_error(void) { return cz::get_error(); }

int cz_init(int device_id, cz_ctx **out) {
  if (!out) return CZ_ERR_INVALID;
  *out = nullptr;
  cz_ctx *ctx = new cz_ctx();
  if (device_id < 0) {  // host-only ctx: container / schedule / weight generation
    *out = ctx;
    return CZ_OK;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0 || device_id >= n) {
    set_error(std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device index out of range"));
    delete ctx;
    return CZ_ERR_NO_DEVICE;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device_id) != cudaSuccess || prop.major != 10) {
    set_error("device is not sm_100 (B200): this library ships sm_100a code only");
    delete ctx;
    return CZ_ERR_NO_DEVICE;
  }
  if (cudaSetDevice(device_id) != cudaSuccess) {
    set_error("cudaSetDevice failed");
    delete ctx;
    return CZ_ERR_CUDA;
  }
  ctx->device = device_id;
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&ctx->prof_ev0) != cudaSuccess || cudaEventCreate(&ctx->prof_ev1) != cudaSuccess ||
      cudaMalloc((void **)&ctx->err_flag_dev, 64) != cudaSuccess || cudaMemset(ctx->err_flag_dev, 0, 64) != cudaSuccess) {
    set_error(std::string("ctx setup failed: ") + cudaGetErrorString(cudaGetLastError()));
    delete ctx;
    return CZ_ERR_CUDA;
  }
  *out = ctx;
  return CZ_OK;
}

void cz_shutdown(cz_ctx *ctx) {
  if (!ctx) return;
  if (ctx->device >= 0) {
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->cdf_stats) cudaFree(ctx->cdf_stats);
    if (ctx->cdf_ecache) cudaFree(ctx->cdf_ecache);
    if (ctx->cdf_eoff) cudaFree(ctx->cdf_eoff);
    if (ctx->err_flag_dev) cudaFree(ctx->err_flag_dev);
    if (ctx->prof_ev0) cudaEventDestroy(ctx->prof_ev0);
    if (ctx->prof_ev1) cudaEventDestroy(ctx->prof_ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  }
  delete ctx;
}

uint64_t cz_launch_count(const cz_ctx *ctx) { return ctx ? ctx->launches : 0; }

int cz_profile_enable(cz_ctx *ctx, int mode) {
  CZ_TRY(require_device(ctx));
  ctx->prof_on = mode == 1;
  ctx->prof_mode = mode;
  return CZ_OK;
}
void *cz_ctx_stream(cz_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
int cz_profile_read(cz_ctx *ctx, double ms_out[CZ_K_FAMILIES], uint64_t launches_out[CZ_K_FAMILIES], int reset) {
  if (!ctx) return CZ_ERR_INVALID;
  if (ctx->ev_used) {  // fold the deferred event pairs in
    cudaStreamSynchronize(ctx->stream);
    for (size_t i = 0; i < ctx->ev_used; i++) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->ev_pool[2 * i], ctx->ev_pool[2 * i + 1]) == cudaSuccess) ctx->prof_ms[ctx->ev_fam[i]] += ms;
    }
    ctx->ev_used = 0;
  }
  for (int i = 0; i < CZ_K_FAMILIES; i++) {
    if (ms_out) ms_out[i] = ctx->prof_ms[i];
    if (launches_out) launches_out[i] = ctx->prof_launches[i];
    if (reset) {
      ctx->prof_ms[i] = 0;
      ctx->prof_launches[i] = 0;
    }
  }
  return CZ_OK;
}

// ---- K1 host-buffer wrappers -------------------------------------------------------------------------------
static int cdf_cols_host(cz_ctx *ctx, int op, const float *logits, size_t V, size_t M, size_t ld, int mode,
                         const uint32_t *arg, uint32_t *sym_out, uint32_t *c_lo, uint32_t *c_hi, double *xe) {
  CZ_TRY(require_device(ctx));
  if (M == 0) return CZ_OK;
  if (!logits || !arg || ld < M) {
    set_error("cdf: null pointer or ld < m");
    return CZ_ERR_INVALID;
  }
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  const size_t b_log = V * ld * sizeof(float), b_u = M * sizeof(uint32_t), b_d = M * sizeof(double);
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  CZ_TRY(ensure_scratch(ctx, al(b_log) + 4 * al(b_u) + al(b_d)));
  char *base = (char *)ctx->scratch;
  float *d_log = (float *)base;
  uint32_t *d_arg = (uint32_t *)(base + al(b_log));
  uint32_t *d_sym = (uint32_t *)((char *)d_arg + al(b_u));
  uint32_t *d_lo = (uint32_t *)((char *)d_sym + al(b_u));
  uint32_t *d_hi = (uint32_t *)((char *)d_lo + al(b_u));
  double *d_xe = (double *)((char *)d_hi + al(b_u));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_log, logits, b_log, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_arg, arg, b_u, cudaMemcpyHostToDevice, ctx->stream));
  CZ_TRY(launch_cdf_cols(ctx, op, mode, d_log, V, M, ld, d_arg, d_sym, d_lo, d_hi, d_xe, ctx->stream));
  if (sym_out) CZ_CUDA_TRY(cudaMemcpyAsync(sym_out, d_sym, b_u, cudaMemcpyDeviceToHost, ctx->stream));
  if (c_lo) CZ_CUDA_TRY(cudaMemcpyAsync(c_lo, d_lo, b_u, cudaMemcpyDeviceToHost, ctx->stream));
  if (c_hi) CZ_CUDA_TRY(cudaMemcpyAsync(c_hi, d_hi, b_u, cudaMemcpyDeviceToHost, ctx->stream));
  if (xe) CZ_CUDA_TRY(cudaMemcpyAsync(xe, d_xe, b_d, cudaMemcpyDeviceToHost, ctx->stream));
  return fetch_device_status(ctx, nullptr, nullptr);
}

int cz_cdf_bounds(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode, const uint32_t *syms,
                  uint32_t *c_lo, uint32_t *c_hi) {
  return cdf_cols_host(ctx, 0, logits, vocab, m, ld, mode, syms, nullptr, c_lo, c_hi, nullptr);
}
int cz_cdf_search(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode, const uint32_t *values,
                  uint32_t *syms_out, uint32_t *c_lo, uint32_t *c_hi) {
  return cdf_cols_host(ctx, 1, logits, vocab, m, ld, mode, values, syms_out, c_lo, c_hi, nullptr);
}
int cz_xe_bits_cols(cz_ctx *ctx, const float *logits, size_t vocab, size_t m, size_t ld, int mode, const uint32_t *syms,
                    double *bits_out) {
  return cdf_cols_host(ctx, 2, logits, vocab, m, ld, mode, syms, nullptr, nullptr, nullptr, bits_out);
}
int cz_cdf_bounds_dev(cz_ctx *ctx, const float *logits_dev, size_t vocab, size_t m, size_t ld, int mode,
                      const uint32_t *syms_dev, uint32_t *c_lo_dev, uint32_t *c_hi_dev) {
  CZ_TRY(require_device(ctx));
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  CZ_TRY(launch_cdf_cols(ctx, 0, mode, logits_dev, vocab, m, ld, syms_dev, nullptr, c_lo_dev, c_hi_dev, nullptr,
                         ctx->stream));
  return fetch_device_status(ctx, nullptr, nullptr);
}
int cz_cdf_full(cz_ctx *ctx, const float *logits, size_t vocab, int mode, uint32_t *cdf_out) {
  CZ_TRY(require_device(ctx));
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  size_t n = (mode == CZ_CDF_RWKV_LITERALS ? vocab + 256 : vocab) + 1;
  size_t b_log = (vocab * sizeof(float) + 255) & ~(size_t)255;
  CZ_TRY(ensure_scratch(ctx, b_log + n * sizeof(uint32_t)));
  float *d_log = (float *)ctx->scratch;
  uint32_t *d_cdf = (uint32_t *)((char *)ctx->scratch + b_log);
  CZ_CUDA_TRY(cudaMemcpyAsync(d_log, logits, vocab * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CZ_TRY(launch_cdf_full(ctx, mode, d_log, vocab, d_cdf, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(cdf_out, d_cdf, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return CZ_OK;
}

// ---- K2 / K3 host-buffer wrappers --------------------------------------------------------------------------
int cz_ac_encode_lanes(cz_ctx *ctx, const uint32_t *c_lo, const uint32_t *c_hi, const uint64_t *lane_off, size_t n_lanes,
                       uint8_t *out, const uint64_t *out_off, uint64_t *out_len) {
  CZ_TRY(require_device(ctx));
  if (n_lanes == 0) return CZ_OK;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  const uint64_t n = lane_off[n_lanes];
  // output capacity: the end of the furthest region
  uint64_t cap = 0;
  for (size_t l = 0; l < n_lanes; l++) {
    uint64_t need = out_off[l] + 4 * (lane_off[l + 1] - lane_off[l]) + 8;
    if (need > cap) cap = need;
  }
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t b_iv = al(n * 4 + 4), b_lane = al((n_lanes + 1) * 8);
  CZ_TRY(ensure_scratch(ctx, 2 * b_iv + 3 * b_lane + al(cap) + 256));
  char *base = (char *)ctx->scratch;
  uint32_t *d_lo = (uint32_t *)base;
  uint32_t *d_hi = (uint32_t *)(base + b_iv);
  uint64_t *d_off = (uint64_t *)(base + 2 * b_iv);
  uint64_t *d_ooff = (uint64_t *)(base + 2 * b_iv + b_lane);
  uint64_t *d_olen = (uint64_t *)(base + 2 * b_iv + 2 * b_lane);
  unsigned long long *d_eidx = (unsigned long long *)(base + 2 * b_iv + 3 * b_lane);
  uint8_t *d_out = (uint8_t *)(base + 2 * b_iv + 3 * b_lane + 256);
  const unsigned long long none = ~0ull;
  CZ_CUDA_TRY(cudaMemcpyAsync(d_lo, c_lo, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_hi, c_hi, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_off, lane_off, (n_lanes + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_ooff, out_off, n_lanes * 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_eidx, &none, 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_TRY(launch_ac_encode_lanes(ctx, d_lo, d_hi, d_off, n_lanes, d_out, d_ooff, d_olen, d_eidx, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(out_len, d_olen, n_lanes * 8, cudaMemcpyDeviceToHost, ctx->stream));
  int rc = fetch_device_status(ctx, d_eidx, nullptr);
  if (rc != CZ_OK) return rc;
  for (size_t l = 0; l < n_lanes; l++)
    CZ_CUDA_TRY(cudaMemcpyAsync(out + out_off[l], d_out + out_off[l], out_len[l], cudaMemcpyDeviceToHost, ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return CZ_OK;
}

int cz_ac_decode_lanes(cz_ctx *ctx, const uint8_t *payload, const uint64_t *pay_off, const uint64_t *pay_len,
                       const uint64_t *lane_off, size_t n_lanes, const uint32_t *cdf, size_t n_sym, uint32_t *syms_out) {
  CZ_TRY(require_device(ctx));
  if (n_lanes == 0) return CZ_OK;
  CZ_CUDA_TRY(cudaSetDevice(ctx->device));
  const uint64_t n = lane_off[n_lanes];
  uint64_t pay_total = 0;
  for (size_t l = 0; l < n_lanes; l++)
    if (pay_off[l] + pay_len[l] > pay_total) pay_total = pay_off[l] + pay_len[l];
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t b_pay = al(pay_total + 1), b_lane = al((n_lanes + 1) * 8), b_cdf = al((n_sym + 1) * 4), b_sym = al(n * 4 + 4);
  CZ_TRY(ensure_scratch(ctx, b_pay + 3 * b_lane + b_cdf + b_sym));
  char *base = (char *)ctx->scratch;
  uint8_t *d_pay = (uint8_t *)base;
  uint64_t *d_poff = (uint64_t *)(base + b_pay);
  uint64_t *d_plen = (uint64_t *)(base + b_pay + b_lane);
  uint64_t *d_loff = (uint64_t *)(base + b_pay + 2 * b_lane);
  uint32_t *d_cdf = (uint32_t *)(base + b_pay + 3 * b_lane);
  uint32_t *d_sym = (uint32_t *)(base + b_pay + 3 * b_lane + b_cdf);
  if (pay_total) CZ_CUDA_TRY(cudaMemcpyAsync(d_pay, payload, pay_total, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_poff, pay_off, n_lanes * 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_plen, pay_len, n_lanes * 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_loff, lane_off, (n_lanes + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(d_cdf, cdf, (n_sym + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
  CZ_TRY(launch_ac_decode_lanes_static(ctx, d_pay, d_poff, d_plen, d_loff, n_lanes, d_cdf, (uint32_t)n_sym, d_sym, ctx->stream));
  CZ_CUDA_TRY(cudaMemcpyAsync(syms_out, d_sym, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CZ_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return CZ_OK;
}

}  // extern "C"
