// Match model (cz_model_set_match, DESIGN.md §6): shared constants, the decoder's per-stream state and the encode stage.
#pragma once
#include "model.h"

namespace cz {

constexpr int kMatchHashBits = 18;    // HB: positions table of 2^18 entries per decode stream
constexpr int kMatchBuckets = 16;     // NB: length buckets, len - K in [0, 16)
constexpr uint32_t kMatchNone = 0xFFFFFFFFu;

// Decoder state of every stream of a cz_decode call, on the device (match_decode_begin clears it):
//   table [S][2^HB]  most recent position p >= K of the stream with each context key (0: none)
//   cnt   [S][32]    tries of bucket b at [b], hits at [16 + b]
//   next  [S][4]     prediction for the stream's next coded token: pred (kMatchNone: none), W, bucket, unused
//   pred_out / w_out per global coded index, when the model has a match-out sink (else nullptr)
struct MatchDecView {
  uint32_t *table = nullptr, *cnt = nullptr, *next = nullptr, *pred_out = nullptr, *w_out = nullptr;
  uint32_t order = 0;
};

// Encode stage, between the model's intervals and the coder lanes: from the model's (c_lo, c_hi) of every coded token (global index)
// builds the list of flag and model intervals the lanes code, and its per-lane offsets.  seg_start_dev: S + 1 offsets (u64).
int match_encode_intervals(cz_model *m, const uint32_t *ids_dev, size_t n_tokens, const uint64_t *seg_start_dev, uint32_t n_segments,
                           const uint32_t *c_lo_dev, const uint32_t *c_hi_dev, cudaStream_t st, const uint32_t **list_lo,
                           const uint32_t **list_hi, const uint64_t **list_lane_off);
// After the lanes coded that list: turns the list indices of the zero-width reports (per lane, lane-relative; the call's smallest)
// back into coded-token indices.
int match_encode_finish(cz_model *m, size_t n_tokens, const uint64_t *seg_start_dev, uint32_t n_segments, unsigned long long *lane_zw_dev,
                        unsigned long long *err_index_dev, cudaStream_t st);
// copies the predictions and weights of the last match_encode_intervals to the match-out sink (async on st) when the model has one
int match_encode_copy_out(cz_model *m, size_t n_tokens, uint32_t n_segments, cudaStream_t st);
// Decoder: reserves and clears the state of n_streams streams; fills *view.
int match_decode_begin(cz_model *m, uint32_t n_streams, size_t n_tokens, cudaStream_t st, MatchDecView *view);
// copies the decoder's match-out arrays to the sink (async on st) when the model has one
int match_decode_end(cz_model *m, size_t n_tokens, cudaStream_t st);

}  // namespace cz
