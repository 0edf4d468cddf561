// Host-side schedule: expands the reference's sequential coding loop into independent CHUNKS.
//
// The reference (src/main.rs:1979, 2275-2290 encode; 2528-2541 decode) walks the token list once and, for the
// SmolLM backend, throws the KV cache away whenever  i > 0 && i % reprime_interval == 0 && index_pos >= eff
// (and i >= reprime_hold_until), re-prefilling the last `eff` tokens.  Between two such points the model state
// depends only on (prime tokens, tokens coded since), so each span is an independent unit of work:
//     chunk = (prime token list P, coded tokens T)   logits for T[j] = model(P ++ T[0..j))[last]
// Gated hint primes (src/main.rs:2123-2149) start a chunk the same way with an explicit prime list.
#include "schedule.h"

#include <algorithm>

namespace cz {

static inline uint32_t eff_context(uint32_t context) { return std::min<uint32_t>(context, 511u); }  // src/main.rs:1935

void build_chunks(uint64_t n_tokens, uint32_t context, uint32_t reprime_interval, const cz_prime_event *events,
                  uint32_t n_events, std::vector<Chunk> &out) {
  out.clear();
  if (n_tokens == 0) return;
  const uint64_t eff = eff_context(context);
  const uint64_t R = reprime_interval ? reprime_interval : 1;
  uint64_t index_pos = 1;  // after step(bos), src/main.rs:1916
  uint64_t hold_until = 0;
  uint32_t ev = 0;
  Chunk cur;
  cur.first = 0;
  cur.n_coded = 0;
  cur.prime_start = 0;
  cur.prime_len = 1;
  cur.event = -1;
  for (uint64_t i = 0; i < n_tokens; i++) {
    bool start_new = false;
    Chunk nc;
    nc.event = -1;
    if (ev < n_events && events[ev].i == i) {  // src/main.rs:1981, 2137/2146
      nc.first = i;
      nc.prime_start = 0;
      nc.prime_len = events[ev].prime_len + (uint32_t)std::min<uint64_t>(events[ev].hist_take, i + 1);  // history tail ++ explicit tokens
      nc.event = (int)ev;
      hold_until = events[ev].hold_until;
      ev++;
      start_new = true;
    }
    if (i < hold_until) {
      // context re-prime suppressed while the hint is meant to stay in the window (src/main.rs:2278)
    } else if (index_pos >= eff && (i % R) == 0 && i > 0) {  // src/main.rs:2280
      const uint64_t end = 1 + i;
      const uint64_t start = end > eff ? end - eff : 0;
      nc.first = i;
      nc.prime_start = start;
      nc.prime_len = (uint32_t)(end - start);
      nc.event = -1;
      start_new = true;
    }
    if (start_new) {
      if (cur.n_coded > 0) out.push_back(cur);
      cur = nc;
      cur.n_coded = 0;
      index_pos = cur.prime_len;
    }
    cur.n_coded++;
    index_pos++;  // step(sym), src/main.rs:2345
  }
  if (cur.n_coded > 0) out.push_back(cur);
}

void build_chunks_prefixed(uint64_t n_tokens, uint64_t n_prefix, uint32_t context, uint32_t reprime_interval, std::vector<Chunk> &out) {
  build_chunks(n_prefix + n_tokens, context, reprime_interval, nullptr, 0, out);
  size_t k = 0;
  for (const Chunk &c : out) {
    if (c.first + c.n_coded <= n_prefix) continue;  // wholly inside the prefix: the next reprime discards its state
    Chunk d = c;
    if (d.first < n_prefix) {  // the chunk in which the prefix ends: its prefix positions join the prime
      const uint64_t skip = n_prefix - d.first;
      d.prime_len += (uint32_t)skip;
      d.n_coded -= (uint32_t)skip;
      d.first = n_prefix;
    }
    d.first -= n_prefix;
    out[k++] = d;
  }
  out.resize(k);
}

}  // namespace cz

extern "C" size_t cz_schedule_chunks_prefixed(uint64_t n_tokens, uint64_t n_prefix, uint32_t context, uint32_t reprime_interval,
                                              uint64_t *first, uint32_t *n_coded, uint64_t *prime_start, uint32_t *prime_len, size_t cap) {
  std::vector<cz::Chunk> chunks;
  cz::build_chunks_prefixed(n_tokens, n_prefix, context, reprime_interval, chunks);
  for (size_t c = 0; c < chunks.size() && c < cap; c++) {
    if (first) first[c] = chunks[c].first;
    if (n_coded) n_coded[c] = chunks[c].n_coded;
    if (prime_start) prime_start[c] = chunks[c].prime_start;
    if (prime_len) prime_len[c] = chunks[c].prime_len;
  }
  return chunks.size();
}

extern "C" size_t cz_schedule_chunks(uint64_t n_tokens, uint32_t context, uint32_t reprime_interval, uint64_t *first,
                                     uint32_t *n_coded, uint64_t *prime_start, uint32_t *prime_len, size_t cap) {
  return cz_schedule_chunks_prefixed(n_tokens, 0, context, reprime_interval, first, n_coded, prime_start, prime_len, cap);
}
