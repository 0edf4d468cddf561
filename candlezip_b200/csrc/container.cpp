// Container format v2 (host-only): byte-compatible with src/main.rs:227-259 (flags), 551-646 (header, LEB128
// varints), 652-677 (AGT2 gate records; legacy AGTB accepted on read, src/main.rs:2469-2484), plus the
// segment-table extension that makes parallel decode possible (DESIGN.md "Container"):
//     flags bit 8 (CZ_FLAG_SEGMENTS) set  =>  after the optional gates section:
//     "SEG1" varint n_segments varint engine { varint n_tokens varint n_bytes } * n_segments
// Files without the bit are exactly the reference's v2 layout (one segment = one AC stream).
// Also a portable BLAKE3 (hash ids are BLAKE3 truncated to 16 bytes, src/main.rs:901-939).
#include <string.h>

#include <vector>

#include "../../include/candlezip_b200.h"

namespace {

size_t put_var(uint8_t *buf, uint64_t v) {  // src/main.rs:566-574
  size_t n = 0;
  while (v >= 0x80) {
    buf[n++] = (uint8_t)((v & 0x7F) | 0x80);
    v >>= 7;
  }
  buf[n++] = (uint8_t)v;
  return n;
}
size_t var_len(uint64_t v) {
  size_t n = 1;
  while (v >= 0x80) {
    v >>= 7;
    n++;
  }
  return n;
}
size_t get_var(const uint8_t *buf, size_t len, uint64_t *out) {  // src/main.rs:576-590
  uint32_t shift = 0;
  uint64_t v = 0;
  size_t n = 0;
  for (;;) {
    if (n >= len) return 0;
    uint8_t b = buf[n++];
    v |= (uint64_t)(b & 0x7F) << shift;
    if (!(b & 0x80)) break;
    shift += 7;
    if (shift > 63) return 0;
  }
  *out = v;
  return n;
}
void put_u32(uint8_t *b, uint32_t v) {
  b[0] = (uint8_t)v;
  b[1] = (uint8_t)(v >> 8);
  b[2] = (uint8_t)(v >> 16);
  b[3] = (uint8_t)(v >> 24);
}
uint32_t get_u32(const uint8_t *b) { return (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24); }

// ---------------- BLAKE3 (portable, single-threaded) ----------------
const uint32_t IV[8] = {0x6A09E667u, 0xBB67AE85u, 0x3C6EF372u, 0xA54FF53Au, 0x510E527Fu, 0x9B05688Cu, 0x1F83D9ABu, 0x5BE0CD19u};
const uint8_t PERM[16] = {2, 6, 3, 10, 7, 0, 4, 13, 1, 11, 12, 5, 9, 14, 15, 8};
enum { CHUNK_START = 1, CHUNK_END = 2, PARENT = 4, ROOT = 8 };
inline uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
inline void gmix(uint32_t *s, int a, int b, int c, int d, uint32_t mx, uint32_t my) {
  s[a] = s[a] + s[b] + mx;
  s[d] = rotr(s[d] ^ s[a], 16);
  s[c] = s[c] + s[d];
  s[b] = rotr(s[b] ^ s[c], 12);
  s[a] = s[a] + s[b] + my;
  s[d] = rotr(s[d] ^ s[a], 8);
  s[c] = s[c] + s[d];
  s[b] = rotr(s[b] ^ s[c], 7);
}
void compress(const uint32_t cv[8], const uint32_t block[16], uint64_t counter, uint32_t block_len, uint32_t flags, uint32_t out[16]) {
  uint32_t s[16] = {cv[0], cv[1], cv[2], cv[3], cv[4], cv[5], cv[6], cv[7], IV[0], IV[1], IV[2], IV[3],
                    (uint32_t)counter, (uint32_t)(counter >> 32), block_len, flags};
  uint32_t m[16];
  memcpy(m, block, 64);
  for (int r = 0; r < 7; r++) {
    gmix(s, 0, 4, 8, 12, m[0], m[1]);
    gmix(s, 1, 5, 9, 13, m[2], m[3]);
    gmix(s, 2, 6, 10, 14, m[4], m[5]);
    gmix(s, 3, 7, 11, 15, m[6], m[7]);
    gmix(s, 0, 5, 10, 15, m[8], m[9]);
    gmix(s, 1, 6, 11, 12, m[10], m[11]);
    gmix(s, 2, 7, 8, 13, m[12], m[13]);
    gmix(s, 3, 4, 9, 14, m[14], m[15]);
    uint32_t p[16];
    for (int i = 0; i < 16; i++) p[i] = m[PERM[i]];
    memcpy(m, p, 64);
  }
  for (int i = 0; i < 8; i++) {
    out[i] = s[i] ^ s[i + 8];
    out[i + 8] = s[i + 8] ^ cv[i];
  }
}
void words_from_bytes(const uint8_t *b, size_t n, uint32_t w[16]) {
  uint8_t tmp[64] = {0};
  memcpy(tmp, b, n);
  for (int i = 0; i < 16; i++) w[i] = get_u32(tmp + 4 * i);
}
// chaining value of one chunk (or, when is_root, the root output words)
void chunk_output(const uint8_t *data, size_t len, uint64_t chunk_idx, bool is_root, uint32_t out[16]) {
  uint32_t cv[8];
  memcpy(cv, IV, 32);
  size_t n_blocks = len == 0 ? 1 : (len + 63) / 64;
  for (size_t b = 0; b < n_blocks; b++) {
    size_t off = b * 64, bl = len - off < 64 ? len - off : 64;
    uint32_t w[16];
    words_from_bytes(data + off, bl, w);
    uint32_t flags = (b == 0 ? CHUNK_START : 0) | (b + 1 == n_blocks ? CHUNK_END : 0);
    if (b + 1 == n_blocks && is_root) flags |= ROOT;
    uint32_t o[16];
    compress(cv, w, b + 1 == n_blocks && is_root ? 0 : chunk_idx, (uint32_t)bl, flags, o);
    if (b + 1 == n_blocks) memcpy(out, o, 64);
    else memcpy(cv, o, 32);
  }
}
void parent_output(const uint32_t l[8], const uint32_t r[8], bool is_root, uint32_t out[16]) {
  uint32_t w[16];
  memcpy(w, l, 32);
  memcpy(w + 8, r, 32);
  compress(IV, w, 0, 64, PARENT | (is_root ? ROOT : 0), out);
}

}  // namespace

extern "C" {

void cz_blake3_16(const uint8_t *data, size_t len, uint8_t out16[16]) {
  uint32_t out[16];
  const size_t n_chunks = len == 0 ? 1 : (len + 1023) / 1024;
  if (n_chunks == 1) {
    // single chunk: the root flag goes on its last block, with the chunk counter 0
    chunk_output(data, len, 0, true, out);
  } else {
    std::vector<uint32_t> stack;  // 8 words per entry
    for (size_t c = 0; c + 1 < n_chunks; c++) {
      uint32_t cv[16];
      chunk_output(data + c * 1024, 1024, c, false, cv);
      uint64_t total = c + 1;
      while ((total & 1) == 0) {
        uint32_t p[16];
        parent_output(&stack[stack.size() - 8], cv, false, p);
        stack.resize(stack.size() - 8);
        memcpy(cv, p, 32);
        total >>= 1;
      }
      stack.insert(stack.end(), cv, cv + 8);
    }
    uint32_t cur[16];
    const size_t last = n_chunks - 1;
    chunk_output(data + last * 1024, len - last * 1024, last, false, cur);
    while (!stack.empty()) {
      uint32_t p[16];
      parent_output(&stack[stack.size() - 8], cur, stack.size() == 8, p);
      stack.resize(stack.size() - 8);
      memcpy(cur, p, 64);
    }
    memcpy(out, cur, 64);
  }
  for (int i = 0; i < 4; i++) put_u32(out16 + 4 * i, out[i]);
}

uint32_t cz_flags_pack(int agent_used, int agent_mock, int gates_present, uint32_t agent_chunk) {  // src/main.rs:247-255
  uint32_t f = 0;
  if (agent_used) f |= CZ_FLAG_AGENT_USED;
  if (agent_mock) f |= CZ_FLAG_AGENT_MOCK;
  if (gates_present) f |= CZ_FLAG_AGENT_GATES;
  f |= (agent_chunk & 0xFFFFu) << 16;
  return f;
}

size_t cz_container_header_size(const cz_header_v2 *h) {
  return 4 + 2 + 4 + var_len(h->token_count) + var_len(h->orig_len_bytes) + 48 + 20 + h->model_file_repr_len;
}

size_t cz_container_write_header(uint8_t *buf, size_t cap, const cz_header_v2 *h, const uint8_t *repr) {  // src/main.rs:592-609
  if (!buf || !h || cap < cz_container_header_size(h)) return 0;
  size_t n = 0;
  put_u32(buf + n, 0x5a505447u);  // "GPTZ"
  n += 4;
  buf[n++] = 2;  // VERSION u16 LE
  buf[n++] = 0;
  put_u32(buf + n, h->bos_token_id);
  n += 4;
  n += put_var(buf + n, h->token_count);
  n += put_var(buf + n, h->orig_len_bytes);
  memcpy(buf + n, h->model_hash16, 16);
  n += 16;
  memcpy(buf + n, h->tokenizer_hash16, 16);
  n += 16;
  memcpy(buf + n, h->orig_hash16, 16);
  n += 16;
  put_u32(buf + n, h->reserved_flags);
  put_u32(buf + n + 4, h->context_window);
  put_u32(buf + n + 8, h->vocab_size);
  put_u32(buf + n + 12, h->model_file_repr_len);
  put_u32(buf + n + 16, h->reprime_interval);
  n += 20;
  if (h->model_file_repr_len) memcpy(buf + n, repr, h->model_file_repr_len);
  n += h->model_file_repr_len;
  return n;
}

size_t cz_container_read_header(const uint8_t *buf, size_t len, cz_header_v2 *h, size_t *repr_off) {  // src/main.rs:611-646
  if (!buf || !h || len < 10) return 0;
  if (get_u32(buf) != 0x5a505447u) return 0;  // bad magic
  if (buf[4] != 2 || buf[5] != 0) return 0;   // bad version
  size_t n = 6, k;
  h->bos_token_id = get_u32(buf + n);
  n += 4;
  if (!(k = get_var(buf + n, len - n, &h->token_count))) return 0;
  n += k;
  if (!(k = get_var(buf + n, len - n, &h->orig_len_bytes))) return 0;
  n += k;
  if (len < n + 68) return 0;
  memcpy(h->model_hash16, buf + n, 16);
  memcpy(h->tokenizer_hash16, buf + n + 16, 16);
  memcpy(h->orig_hash16, buf + n + 32, 16);
  n += 48;
  h->reserved_flags = get_u32(buf + n);
  h->context_window = get_u32(buf + n + 4);
  h->vocab_size = get_u32(buf + n + 8);
  h->model_file_repr_len = get_u32(buf + n + 12);
  h->reprime_interval = get_u32(buf + n + 16);
  n += 20;
  if (h->model_file_repr_len > len - n) return 0;  // (not `len < n + repr_len`: an untrusted length must not be added to an offset)
  if (repr_off) *repr_off = n;
  return n + h->model_file_repr_len;
}

size_t cz_container_write_gates(uint8_t *buf, size_t cap, const uint8_t *records, size_t n) {  // src/main.rs:658-670
  const size_t need = 4 + var_len(n) + n;
  if (!buf || cap < need) return 0;
  memcpy(buf, "AGT2", 4);
  size_t k = 4 + put_var(buf + 4, n);
  for (size_t i = 0; i < n; i++) buf[k + i] = records[i] & 0x1F;  // gate | cand<<1 | budget<<3
  return need;
}

size_t cz_container_read_gates(const uint8_t *buf, size_t len, uint8_t *records, size_t cap, size_t *n_records) {
  if (!buf || len < 5) return 0;
  uint64_t cnt;
  size_t k = get_var(buf + 4, len - 4, &cnt);
  if (!k) return 0;
  size_t n = 4 + k;
  // `cnt` is an untrusted 64-bit varint: compare it against what is LEFT (n <= len here), never add it to an offset -- a count
  // near 2^64 wraps `n + cnt` / `(cnt + 7) / 8` and would let the copy loops below run past the buffer
  if (!memcmp(buf, "AGT2", 4)) {  // src/main.rs:2472-2476
    if (cnt > len - n) return 0;
    for (uint64_t i = 0; i < cnt && i < cap; i++) records[i] = buf[n + i] & 0x1F;
    if (n_records) *n_records = (size_t)cnt;
    return n + (size_t)cnt;
  }
  if (!memcmp(buf, "AGTB", 4)) {  // legacy bit vector, src/main.rs:2477-2482: gate bit only, candidate 0 / budget 2 (2554)
    if (cnt / 8 > len - n) return 0;
    const size_t nbytes = (size_t)(cnt / 8 + (cnt % 8 ? 1 : 0));
    if (nbytes > len - n) return 0;
    for (uint64_t i = 0; i < cnt && i < cap; i++) {
      uint8_t g = (buf[n + i / 8] >> (i % 8)) & 1;
      records[i] = (uint8_t)(g | (0 << 1) | (2 << 3));
    }
    if (n_records) *n_records = (size_t)cnt;
    return n + nbytes;
  }
  return 0;
}

size_t cz_container_write_segments(uint8_t *buf, size_t cap, int engine, const uint64_t *seg_tokens, const uint64_t *seg_bytes,
                                   size_t n) {
  size_t need = 4 + var_len(n) + var_len((uint64_t)engine);
  for (size_t i = 0; i < n; i++) need += var_len(seg_tokens[i]) + var_len(seg_bytes[i]);
  if (!buf || cap < need) return 0;
  memcpy(buf, "SEG1", 4);
  size_t k = 4;
  k += put_var(buf + k, n);
  k += put_var(buf + k, (uint64_t)engine);
  for (size_t i = 0; i < n; i++) {
    k += put_var(buf + k, seg_tokens[i]);
    k += put_var(buf + k, seg_bytes[i]);
  }
  return k;
}

size_t cz_container_read_segments(const uint8_t *buf, size_t len, int *engine, uint64_t *seg_tokens, uint64_t *seg_bytes, size_t cap,
                                  size_t *n_out) {
  if (!buf || len < 6 || memcmp(buf, "SEG1", 4)) return 0;
  size_t k = 4, r;
  uint64_t n, eng;
  if (!(r = get_var(buf + k, len - k, &n))) return 0;
  k += r;
  if (!(r = get_var(buf + k, len - k, &eng))) return 0;
  k += r;
  if (n > (len - k) / 2) return 0;  // every entry takes at least two bytes: an untrusted count cannot exceed what is left
  uint64_t total_bytes = 0;
  for (uint64_t i = 0; i < n; i++) {
    uint64_t a, b;
    if (!(r = get_var(buf + k, len - k, &a))) return 0;
    k += r;
    if (!(r = get_var(buf + k, len - k, &b))) return 0;
    k += r;
    if (b > len || total_bytes > len - b) return 0;  // the segments' byte counts cannot add up to more than the file holds
    total_bytes += b;
    if (i < cap) {
      if (seg_tokens) seg_tokens[i] = a;
      if (seg_bytes) seg_bytes[i] = b;
    }
  }
  if (engine) *engine = (int)eng;
  if (n_out) *n_out = (size_t)n;
  return k;
}

size_t cz_container_write_dictionary(uint8_t *buf, size_t cap, uint64_t n_symbols, const uint8_t hash16[16]) {
  const size_t need = 4 + var_len(n_symbols) + 16;
  if (!buf || !hash16 || cap < need) return 0;
  memcpy(buf, "DIC1", 4);
  size_t k = 4 + put_var(buf + 4, n_symbols);
  memcpy(buf + k, hash16, 16);
  return k + 16;
}

size_t cz_container_read_dictionary(const uint8_t *buf, size_t len, uint64_t *n_symbols, uint8_t hash16[16]) {
  if (!buf || len < 5 || memcmp(buf, "DIC1", 4)) return 0;
  uint64_t n;
  const size_t r = get_var(buf + 4, len - 4, &n);
  if (!r || n == 0) return 0;  // an empty dictionary is written as no section at all
  const size_t k = 4 + r;
  if (len - k < 16) return 0;
  if (n_symbols) *n_symbols = n;
  if (hash16) memcpy(hash16, buf + k, 16);
  return k + 16;
}

size_t cz_container_write_match(uint8_t *buf, size_t cap, uint32_t order) {
  if (!buf || order < 1 || order > 16 || cap < 4 + var_len(order)) return 0;
  memcpy(buf, "MAT1", 4);
  return 4 + put_var(buf + 4, order);
}

size_t cz_container_read_match(const uint8_t *buf, size_t len, uint32_t *order) {
  if (!buf || len < 5 || memcmp(buf, "MAT1", 4)) return 0;
  uint64_t k;
  const size_t r = get_var(buf + 4, len - 4, &k);
  if (!r || k < 1 || k > 16) return 0;
  if (order) *order = (uint32_t)k;
  return 4 + r;
}

}  // extern "C"
