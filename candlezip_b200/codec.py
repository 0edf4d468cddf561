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
from .api import split_segments


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


def _check_policy(on_zero_width):
    if on_zero_width not in ("stored", "floor"):
        raise ValueError(f"on_zero_width must be 'stored' or 'floor', not {on_zero_width!r}")


def tokenize(model, data: bytes, tokenizer):
    """the coded symbols of `data`: token ids, plus RWKV-7's literal escapes with an RwkvTokenizer"""
    if model.cfg.get("arch", 0) == 1 and isinstance(tokenizer, RwkvTokenizer):
        return plan_rwkv_symbols(data, tokenizer, int(model.cfg["vocab"]))
    return tokenizer.encode_bytes(data)


def header_fields(model, data: bytes, n_tokens, bos, context, reprime_interval, model_hash16, tokenizer_hash16):
    return dict(bos_token_id=bos, token_count=n_tokens, orig_len_bytes=len(data), model_hash16=model_hash16,
                tokenizer_hash16=tokenizer_hash16, orig_hash16=container.blake3_16(data), context_window=context,
                vocab_size=int(model.cfg["vocab"]), reprime_interval=reprime_interval, reserved_flags=0)


def stored_container(fields, model_repr, data: bytes) -> bytes:
    return container.write_container(dict(fields, reserved_flags=_lib.CZ_FLAG_STORED), model_repr, [bytes(data)])


def coded_container(model, fields, model_repr, pays, seg) -> bytes:
    """one payload: the reference's v2 layout; several: the SEG1 table"""
    seg_tokens = np.diff(seg) if len(pays) > 1 else None
    return container.write_container(fields, model_repr, pays, seg_tokens=seg_tokens, engine=model.engine)


def compress(model, data: bytes, tokenizer=None, n_segments=1, bos=0, context=512, reprime_interval=512, model_repr=b"model.safetensors",
             model_hash16=b"\0" * 16, tokenizer_hash16=b"\0" * 16, on_zero_width="stored"):
    """bytes -> .canz container bytes.  n_segments == 1 gives the reference's v2 layout (header | payload).
    on_zero_width: what to do when the SmolLM coder meets a token it cannot code (CZ_ERR_ZERO_WIDTH): "stored" writes the bytes
    uncoded (CZ_FLAG_STORED), "floor" codes the whole input again with the floored pdf (CZ_FLAG_PDF_FLOOR).  An input that codes
    without such a token gives the same container either way."""
    _check_policy(on_zero_width)
    tokenizer = tokenizer or ByteTokenizer()
    ids = tokenize(model, data, tokenizer)
    fields = header_fields(model, data, len(ids), bos, context, reprime_interval, model_hash16, tokenizer_hash16)
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
            return stored_container(fields, model_repr, data)
    return coded_container(model, fields, model_repr, pays, seg)


class _Parsed:
    """one container, read and checked up to the point where its payloads need the model"""

    def __init__(self, f, pays=None, seg=None, key=None, data=None):
        self.f, self.pays, self.seg, self.key, self.data = f, pays, seg, key, data


def _parse(model, blob: bytes, verify) -> _Parsed:
    f, _, gates, _, seg_tokens, pays = container.read_container(blob)
    n = int(f["token_count"])
    pdf_floor = bool(f["reserved_flags"] & _lib.CZ_FLAG_PDF_FLOOR)
    if pdf_floor and (f["reserved_flags"] & _lib.CZ_FLAG_STORED or model.cfg.get("arch", 0) == 1):
        raise ValueError("PDF_FLOOR marks a SmolLM payload coded with the floored pdf: invalid with STORED or on an RWKV-7 model")
    if f["reserved_flags"] & _lib.CZ_FLAG_STORED:
        data = b"".join(pays)
        if len(data) != int(f["orig_len_bytes"]) or (verify and container.blake3_16(data) != f["orig_hash16"]):
            raise ValueError("stored payload does not match the header")
        return _Parsed(f, data=data)
    if gates is not None:
        raise ValueError("gated containers are decoded through gate.events_from_records + Model.decode(events=...)")
    seg = np.concatenate([[0], np.cumsum(seg_tokens)]).astype(np.uint64) if seg_tokens is not None else np.array([0, n], np.uint64)
    if int(seg[-1]) != n:
        raise ValueError("segment table does not add up to token_count")
    key = (int(f["bos_token_id"]), int(f["context_window"]), int(f["reprime_interval"]), pdf_floor)
    return _Parsed(f, pays=pays, seg=seg, key=key)


def _finish(model, tokenizer, f, ids, verify) -> bytes:
    """decoded symbols -> bytes, checked against the header"""
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


def decompress(model, blob: bytes, tokenizer=None, verify=True) -> bytes:
    tokenizer = tokenizer or ByteTokenizer()
    p = _parse(model, blob, verify)
    if p.data is not None:
        return p.data
    bos, context, reprime_interval, pdf_floor = p.key
    ids = model.decode(p.pays, p.seg, bos=bos, context=context, reprime_interval=reprime_interval, pdf_floor=pdf_floor)
    return _finish(model, tokenizer, p.f, ids, verify)


# ---- many files per call ----------------------------------------------------------------------------------------------------------
# The GPU path earns its speed from batching independent streams: every kernel is row-invariant, so a segment's bytes do not depend on
# what else is in the batch.  compress_many / decompress_many pack the segments of many files into one cz_encode call and into
# lock-step cz_decode waves; the planning below is pure (the coding calls are injected) so that it is testable without a GPU.

def pack_segments(lengths, n_segments):
    """files of lengths[i] tokens, each split into segments as compress() splits it, laid end to end.
    Returns (seg_start of the concatenation, [(g0, g1)] global segment range of each file, [file-local seg_start])."""
    local = [split_segments(int(n), n_segments) for n in lengths]
    starts, ranges, off = [0], [], 0
    for loc in local:
        g0 = len(starts) - 1
        starts.extend(off + int(x) for x in loc[1:])
        off += int(loc[-1])
        ranges.append((g0, len(starts) - 1))
    return np.asarray(starts, np.uint64), ranges, local


def zero_width_files(ranges, first_zw):
    """indices of the files with at least one segment that reported a zero-width token (first_zw: per global segment, or None)"""
    if first_zw is None:
        return []
    first_zw = np.asarray(first_zw, np.uint64)
    return [i for i, (g0, g1) in enumerate(ranges) if np.any(first_zw[g0:g1] != np.uint64(_lib.NO_ZERO_WIDTH))]


def encode_many(id_lists, n_segments, encode_fn, on_zero_width="stored"):
    """encode_fn(ids, seg_start, pdf_floor) -> (per-segment payloads, per-segment first zero-width index or None).
    All files go through ONE call (pdf_floor False).  The files with a zero-width token are then, by the policy, either marked STORED
    or re-coded together in ONE more call with pdf_floor True.  Returns per file (payloads or None, file-local seg_start, flag) with
    flag 0, CZ_FLAG_PDF_FLOOR or CZ_FLAG_STORED."""
    _check_policy(on_zero_width)

    def run(files, pdf_floor):
        ids = np.concatenate([np.asarray(id_lists[i], np.uint32) for i in files]).astype(np.uint32)
        seg, ranges, local = pack_segments([len(id_lists[i]) for i in files], n_segments)
        pays, first_zw = encode_fn(ids, seg, pdf_floor)
        assert len(pays) == len(seg) - 1
        coded = {i: (list(pays[g0:g1]), loc) for i, (g0, g1), loc in zip(files, ranges, local)}
        return coded, [files[k] for k in zero_width_files(ranges, first_zw)]

    out = [None] * len(id_lists)
    if not id_lists:
        return out
    coded, bad = run(list(range(len(id_lists))), False)
    for i, (pays, loc) in coded.items():
        out[i] = (pays, loc, 0)
    if bad and on_zero_width == "floor":
        coded, again = run(bad, True)
        if again:
            raise RuntimeError(f"files {again} met a zero-width token under the floored pdf")
        for i, (pays, loc) in coded.items():
            out[i] = (pays, loc, _lib.CZ_FLAG_PDF_FLOOR)
    elif bad:
        for i in bad:
            out[i] = (None, out[i][1], _lib.CZ_FLAG_STORED)
    return out


def compress_many(model, datas, tokenizer=None, n_segments=1, bos=0, context=512, reprime_interval=512, model_repr=b"model.safetensors",
                  model_hash16=b"\0" * 16, tokenizer_hash16=b"\0" * 16, on_zero_width="stored"):
    """[bytes] -> [container bytes], element i equal byte for byte to compress(model, datas[i], <same arguments>).  The segments of all
    files are coded in one Model.encode call with the per-segment zero-width report on; the files that report a zero-width token get
    the on_zero_width fallback (all "floor" files in one more call)."""
    _check_policy(on_zero_width)
    tokenizer = tokenizer or ByteTokenizer()
    id_lists = [tokenize(model, d, tokenizer) for d in datas]

    def encode_fn(ids, seg_start, pdf_floor):
        # the sink is set on the floored call too: no token can be zero-width there, and encode_many checks that none was
        pays, _, first_zw = model.encode(ids, seg_start=seg_start, bos=bos, context=context, reprime_interval=reprime_interval,
                                         pdf_floor=pdf_floor, zero_width_out=True)
        return pays, first_zw

    out = []
    for i, (data, ids, (pays, loc, flag)) in enumerate(zip(datas, id_lists, encode_many(id_lists, n_segments, encode_fn, on_zero_width))):
        fields = header_fields(model, data, len(ids), bos, context, reprime_interval, model_hash16, tokenizer_hash16)
        if flag == _lib.CZ_FLAG_STORED:
            sys.stderr.write(f"candlezip_b200: file {i}: zero-width coding interval; writing a STORED container\n")
            out.append(stored_container(fields, model_repr, data))
            continue
        if flag == _lib.CZ_FLAG_PDF_FLOOR:
            sys.stderr.write(f"candlezip_b200: file {i}: zero-width coding interval; coded with the floored pdf\n")
        out.append(coded_container(model, dict(fields, reserved_flags=flag), model_repr, pays, loc))
    return out


def decode_waves(jobs, max_streams):
    """jobs[i]: None (nothing to decode) or (key, segment lengths) of file i.  Segments of files with the same key (bos, context,
    reprime_interval, pdf_floor) share calls; within a key they are sorted by length, longest first (stable), which is the lock-step
    decoder's precondition, and cut into waves of at most max_streams.  Zero-length segments decode to nothing and are left out.
    Returns [(key, [(file, segment, length)])], one entry per decode call."""
    if max_streams < 1:
        raise ValueError("max_streams must be >= 1")
    groups = {}
    for f, job in enumerate(jobs):
        if job is None:
            continue
        key, lens = job
        groups.setdefault(key, []).extend((f, g, int(n)) for g, n in enumerate(lens) if int(n) > 0)
    waves = []
    for key, items in groups.items():
        items.sort(key=lambda t: -t[2])
        waves += [(key, items[k : k + max_streams]) for k in range(0, len(items), max_streams)]
    return waves


def decode_many(jobs, payloads, decode_fn, max_streams):
    """jobs as decode_waves; payloads[i]: file i's per-segment payloads.  decode_fn(key, payloads, seg_start) -> ids of the
    concatenated segments.  Returns per file its ids in segment order (None where jobs[i] is None)."""
    parts = [None if job is None else [np.zeros(0, np.uint32)] * len(job[1]) for job in jobs]
    for key, items in decode_waves(jobs, max_streams):
        seg = np.concatenate([[0], np.cumsum([n for _, _, n in items])]).astype(np.uint64)
        ids = np.asarray(decode_fn(key, [payloads[f][g] for f, g, _ in items], seg), np.uint32)
        assert ids.shape[0] == int(seg[-1])
        for (f, g, _), a, b in zip(items, seg[:-1], seg[1:]):
            parts[f][g] = ids[int(a) : int(b)]
    return [None if p is None else np.concatenate(p).astype(np.uint32) for p in parts]


def decompress_many(model, blobs, tokenizer=None, max_streams=2048, verify=True) -> list:
    """[container bytes] -> [bytes], element i equal to decompress(model, blobs[i], tokenizer).  STORED containers and empty files need
    no GPU work; the segments of all other containers are decoded in lock-step waves of at most max_streams streams (decode_waves).
    The default of 2,048 streams decodes at nearly the 4,096-stream rate with half the KV memory (48 GB for SmolLM-135M), and lets a
    container with more segments than one cz_decode call could hold decode too.  A gated (AGT2) container, a bad header or a hash
    mismatch raises ValueError naming the index of the blob."""
    tokenizer = tokenizer or ByteTokenizer()
    parsed = []
    for i, blob in enumerate(blobs):
        try:
            parsed.append(_parse(model, blob, verify))
        except ValueError as e:
            raise ValueError(f"blob {i}: {e}") from None
    jobs = [None if p.data is not None or int(p.f["token_count"]) == 0 else (p.key, np.diff(p.seg)) for p in parsed]

    def decode_fn(key, pays, seg_start):
        bos, context, reprime_interval, pdf_floor = key
        return model.decode(pays, seg_start, bos=bos, context=context, reprime_interval=reprime_interval, pdf_floor=pdf_floor)

    ids = decode_many(jobs, [p.pays for p in parsed], decode_fn, max_streams)
    out = []
    for i, (p, x) in enumerate(zip(parsed, ids)):
        if p.data is not None:
            out.append(p.data)
            continue
        try:
            out.append(_finish(model, tokenizer, p.f, np.zeros(0, np.uint32) if x is None else x, verify))
        except ValueError as e:
            raise ValueError(f"blob {i}: {e}") from None
    return out
