#pragma once
#include <stdint.h>

#include <vector>

#include "../../include/candlezip_b200.h"

namespace cz {

// One independent unit of model work.  Indices are relative to ONE segment whose token sequence is
// S = [bos, t_0 .. t_{n-1}]  (S[k] is the reference's ids[k]).
struct Chunk {
  uint64_t first;        // coded index i of the first coded token (codes t_first .. t_{first+n_coded-1})
  uint32_t n_coded;
  uint64_t prime_start;  // prime = S[prime_start .. prime_start + prime_len) unless event >= 0
  uint32_t prime_len;
  int event;             // >= 0: prime is events[event].prime (explicit token list)
};

void build_chunks(uint64_t n_tokens, uint32_t context, uint32_t reprime_interval, const cz_prime_event *events,
                  uint32_t n_events, std::vector<Chunk> &out);
// The chunks of the last n_tokens of a segment S = [bos, p_0 .. p_{n_prefix-1}, t_0 .. t_{n-1}] whose first n_prefix coded
// positions are a dictionary that is never coded: build_chunks over n_prefix + n_tokens, chunks wholly inside the prefix dropped, the
// prefix positions of the chunk in which the prefix ends moved into its prime.  `first` counts from t_0; `prime_start` indexes S.
void build_chunks_prefixed(uint64_t n_tokens, uint64_t n_prefix, uint32_t context, uint32_t reprime_interval, std::vector<Chunk> &out);

}  // namespace cz
