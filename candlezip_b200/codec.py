"""File-level compress / decompress over the batched hot path (host side, once per file; SURVEY 8 f-1 / f-2).

  reference                                                        here
  ---------------------------------------------------------------  ---------------------------------------------------
  Tokenizer::{new, encode_bytes, decode_bytes}  (candle_rwkv7/     RwkvTokenizer (same table construction: per 2-byte prefix,
      src/models/rwkv7.rs:546-610): first match in descending       descending id; first prefix match wins)
      id order among the tokens sharing the first two bytes
  plan_rwkv_symbols / rwkv_detok_with_literals                      plan_rwkv_symbols / rwkv_detok_with_literals: tokens, then
      (src/main.rs:833-895): literal-escape symbols V + byte          literal escapes for whatever the vocabulary cannot cover
  SmolLM: tok.encode(from_utf8_lossy(data)) (main.rs:1850-1857)     ByteTokenizer (id = byte) when no tokenizer.json exists
      -- lossy for non-UTF-8 input                                   offline: byte-exact for EVERY input (SURVEY 7.3c)
  encode_file / decode_file container assembly (1793-2405,         compress() / decompress(): header v2 (+ SEG1 segment table,
      2407-2660)                                                     + AGT2 gates), BLAKE3-128 ids, orig hash VERIFIED on decode
"""
import json
import sys

import numpy as np

from . import _lib, container


class ByteTokenizer:
    """identity tokenisation: one token per byte (ids 0..255).  Lossless for every input."""
    vocab_size = 256

    def encode_bytes(self, data: bytes):
        return np.frombuffer(data, np.uint8).astype(np.uint32)

    def decode_bytes(self, ids):
        return bytes(np.asarray(ids, np.uint32).astype(np.uint8))


class RwkvTokenizer:
    """RWKV "world" trie tokenizer exactly as candle_rwkv7/src/models/rwkv7.rs:553-608."""

    def __init__(self, token2idx: dict):
        self.token2idx = {bytes(k): int(v) for k, v in token2idx.items()}
        self.idx2token = {v: k for k, v in self.token2idx.items()}
        self.table = {}
        for idx in sorted(self.idx2token, reverse=True):  # descending id (rwkv7.rs:566)
            s = self.idx2token[idx]
            if len(s) >= 2:
                self.table.setdefault((s[0], s[1]), []).append(s)

    @classmethod
    def from_json(cls, path):
        with open(path, "r", encoding="utf-8") as f:
            return cls({k.encode("utf-8"): v for k, v in json.load(f).items()})

    def encode_bytes(self, data: bytes):
        out, i, n = [], 0, len(data)
        while i < n:
            s = data[i:i + 1]
            if i + 1 < n:
                for cand in self.table.get((data[i], data[i + 1]), ()):
                    if data.startswith(cand, i):
                        s = cand
                        break
            i += len(s)
            tok = self.token2idx.get(s)
            if tok is None:  # rwkv7.rs:595-601: a lossless coder cannot substitute a fallback token
                raise KeyError(f"tokenizer vocabulary missing byte sequence {s!r}")
            out.append(tok)
        return np.asarray(out, np.uint32)

    def decode_bytes(self, ids):
        return b"".join(self.idx2token.get(int(t), b"") for t in ids)


def plan_rwkv_symbols(data: bytes, tok: RwkvTokenizer, vocab_size: int):
    """src/main.rs:833-864: token ids, or literal-escape symbols vocab_size + byte for what the vocabulary cannot express"""
    try:
        ids = tok.encode_bytes(data)
    except KeyError:
        return (vocab_size + np.frombuffer(data, np.uint8).astype(np.uint32)).astype(np.uint32)
    covered = sum(len(tok.idx2token[int(t)]) for t in ids)
    if covered < len(data):
        tail = vocab_size + np.frombuffer(data[covered:], np.uint8).astype(np.uint32)
        ids = np.concatenate([ids, tail]).astype(np.uint32)
    return ids


def rwkv_detok_with_literals(tok: RwkvTokenizer, symbols, vocab_size: int) -> bytes:
    """src/main.rs:866-895"""
    out = bytearray()
    for s in symbols:
        s = int(s)
        out += tok.idx2token.get(s, b"") if s < vocab_size else bytes([s - vocab_size])
    return bytes(out)


def compress(model, data: bytes, tokenizer=None, n_segments=1, bos=0, context=512, reprime_interval=512, model_repr=b"model.safetensors",
             model_hash16=b"\0" * 16, tokenizer_hash16=b"\0" * 16, on_zero_width="stored"):
    """bytes -> .canz container bytes.  n_segments == 1 gives the reference's v2 layout (header | payload).
    on_zero_width: what to do when the SmolLM coder meets a token it cannot code (CZ_ERR_ZERO_WIDTH): "stored" writes the bytes
    uncoded (CZ_FLAG_STORED), "floor" codes the whole input again with the floored pdf (CZ_FLAG_PDF_FLOOR).  An input that codes
    without such a token gives the same container either way."""
    if on_zero_width not in ("stored", "floor"):
        raise ValueError(f"on_zero_width must be 'stored' or 'floor', not {on_zero_width!r}")
    tokenizer = tokenizer or ByteTokenizer()
    vocab = int(model.cfg["vocab"])
    if model.cfg.get("arch", 0) == 1:
        ids = plan_rwkv_symbols(data, tokenizer, vocab) if isinstance(tokenizer, RwkvTokenizer) else tokenizer.encode_bytes(data)
    else:
        ids = tokenizer.encode_bytes(data)
    fields = dict(bos_token_id=bos, token_count=len(ids), orig_len_bytes=len(data), model_hash16=model_hash16,
                  tokenizer_hash16=tokenizer_hash16, orig_hash16=container.blake3_16(data), context_window=context, vocab_size=vocab,
                  reprime_interval=reprime_interval, reserved_flags=0)
    try:
        pays, seg = model.encode(ids, n_segments=n_segments, bos=bos, context=context, reprime_interval=reprime_interval)
    except _lib.CzError as e:
        if e.code != _lib.CZ_ERR_ZERO_WIDTH:
            raise
        # SmolLM coding has no probability floor (src/main.rs:2295): a token whose mass quantises to a zero-width interval cannot be
        # coded -- the reference writes a corrupt stream there (SURVEY 7.3a).  Every input must still round-trip: either code it with
        # the floored pdf (softmax_pdf_floor, src/main.rs:758-767, under which no token is zero-width) or store the bytes uncoded
        # (the message names the offending token index for whoever wants to know why).
        if on_zero_width == "floor":
            sys.stderr.write(f"candlezip_b200: {e}; coding with the floored pdf\n")
            pays, seg = model.encode(ids, n_segments=n_segments, bos=bos, context=context, reprime_interval=reprime_interval, pdf_floor=True)
            fields["reserved_flags"] = _lib.CZ_FLAG_PDF_FLOOR
        else:
            sys.stderr.write(f"candlezip_b200: {e}; writing a STORED container\n")
            return container.write_container(dict(fields, reserved_flags=_lib.CZ_FLAG_STORED), model_repr, [bytes(data)])
    seg_tokens = np.diff(seg) if len(pays) > 1 else None
    return container.write_container(fields, model_repr, pays, seg_tokens=seg_tokens, engine=model.engine)


def decompress(model, blob: bytes, tokenizer=None, verify=True) -> bytes:
    tokenizer = tokenizer or ByteTokenizer()
    f, _, gates, _, seg_tokens, pays = container.read_container(blob)
    n = int(f["token_count"])
    pdf_floor = bool(f["reserved_flags"] & _lib.CZ_FLAG_PDF_FLOOR)
    if pdf_floor and (f["reserved_flags"] & _lib.CZ_FLAG_STORED or model.cfg.get("arch", 0) == 1):
        raise ValueError("PDF_FLOOR marks a SmolLM payload coded with the floored pdf: invalid with STORED or on an RWKV-7 model")
    if f["reserved_flags"] & _lib.CZ_FLAG_STORED:
        data = b"".join(pays)
        if len(data) != int(f["orig_len_bytes"]) or (verify and container.blake3_16(data) != f["orig_hash16"]):
            raise ValueError("stored payload does not match the header")
        return data
    if gates is not None:
        raise ValueError("gated containers are decoded through gate.events_from_records + Model.decode(events=...)")
    seg = np.concatenate([[0], np.cumsum(seg_tokens)]).astype(np.uint64) if seg_tokens is not None else np.array([0, n], np.uint64)
    if int(seg[-1]) != n:
        raise ValueError("segment table does not add up to token_count")
    ids = model.decode(pays, seg, bos=int(f["bos_token_id"]), context=int(f["context_window"]), reprime_interval=int(f["reprime_interval"]),
                       pdf_floor=pdf_floor)
    vocab = int(model.cfg["vocab"])
    if model.cfg.get("arch", 0) == 1 and isinstance(tokenizer, RwkvTokenizer):
        data = rwkv_detok_with_literals(tokenizer, ids, vocab)
    else:
        data = tokenizer.decode_bytes(ids)
    # the reference writes orig_hash16 (main.rs:2370) but never checks it on decode (SURVEY 5): here it is verified
    if verify and container.blake3_16(data) != f["orig_hash16"]:
        raise ValueError("decoded bytes do not match the container's BLAKE3-128 of the original")
    if len(data) != int(f["orig_len_bytes"]):
        raise ValueError("decoded length differs from the header")
    return data
