"""Container v2 (+ segment-table and dictionary extensions) over the C ABI: src/main.rs:227-259, 551-677."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import lib

CZ_FLAG_SEGMENTS = _lib.CZ_FLAG_SEGMENTS
CZ_FLAG_DICTIONARY = _lib.CZ_FLAG_DICTIONARY
CZ_FLAG_MATCH = _lib.CZ_FLAG_MATCH


def blake3_16(data: bytes) -> bytes:
    buf = (C.c_uint8 * max(1, len(data))).from_buffer_copy(data or b"\0")
    out = (C.c_uint8 * 16)()
    lib.cz_blake3_16(buf, len(data), out)
    return bytes(out)


def dictionary_id(symbols):
    """(n_symbols, BLAKE3-128 of the symbols as little-endian u32): what a DIC1 section records of a dictionary"""
    a = np.asarray(symbols, np.uint32)
    return int(a.shape[0]), blake3_16(a.astype("<u4").tobytes())


def _hdr(fields: dict, repr_len: int):
    h = _lib.HeaderV2()
    h.bos_token_id = fields.get("bos_token_id", 0)
    h.token_count = fields["token_count"]
    h.orig_len_bytes = fields["orig_len_bytes"]
    for name in ("model_hash16", "tokenizer_hash16", "orig_hash16"):
        v = fields.get(name, b"\0" * 16)
        getattr(h, name)[:] = list(v)
    h.reserved_flags = fields.get("reserved_flags", 0)
    h.context_window = fields.get("context_window", 512)
    h.vocab_size = fields["vocab_size"]
    h.model_file_repr_len = repr_len
    h.reprime_interval = fields.get("reprime_interval", 512)
    return h


def write_container(fields: dict, model_file_repr: bytes, payloads, seg_tokens=None, gates=None, engine=0, dictionary=None,
                    match_order=0) -> bytes:
    """One payload and no seg_tokens -> byte-identical layout to the reference (header | [AGT2] | payload).
    dictionary: dictionary_id() of the dictionary the payloads were coded with (CZ_FLAG_DICTIONARY + a DIC1 section), or None.
    match_order: the match model's order the payloads were coded with (CZ_FLAG_MATCH + a MAT1 section), or 0."""
    flags = fields.get("reserved_flags", 0)
    if dictionary is not None:
        if flags & _lib.CZ_FLAG_STORED:
            raise ValueError("a STORED payload is not coded: it has no dictionary")
        flags |= CZ_FLAG_DICTIONARY
    if match_order:
        if flags & _lib.CZ_FLAG_STORED:
            raise ValueError("a STORED payload is not coded: it has no match model")
        if not 1 <= int(match_order) <= 16:
            raise ValueError(f"match order {match_order} is outside [1, 16]")
        flags |= CZ_FLAG_MATCH
    segmented = seg_tokens is not None and len(payloads) >= 1 and not (len(payloads) == 1 and seg_tokens is None)
    if seg_tokens is not None:
        flags |= CZ_FLAG_SEGMENTS
    if gates is not None:
        flags |= 1 << 2
    fields = dict(fields, reserved_flags=flags)
    h = _hdr(fields, len(model_file_repr))
    cap = int(lib.cz_container_header_size(C.byref(h))) + 64
    buf = (C.c_uint8 * cap)()
    rp = (C.c_uint8 * max(1, len(model_file_repr))).from_buffer_copy(model_file_repr or b"\0")
    n = lib.cz_container_write_header(buf, cap, C.byref(h), rp)
    assert n, "header write failed"
    out = bytearray(bytes(buf[:n]))
    if gates is not None:
        g = (C.c_uint8 * max(1, len(gates)))(*gates)
        gb = (C.c_uint8 * (len(gates) + 16))()
        k = lib.cz_container_write_gates(gb, len(gates) + 16, g, len(gates))
        out += bytes(gb[:k])
    if segmented:
        st = np.asarray(seg_tokens, np.uint64)
        sb = np.asarray([len(p) for p in payloads], np.uint64)
        sbuf = (C.c_uint8 * (32 + 20 * len(payloads)))()
        k = lib.cz_container_write_segments(sbuf, len(sbuf), engine, st.ctypes.data_as(_lib.u64p), sb.ctypes.data_as(_lib.u64p), len(payloads))
        assert k, "segment table write failed"
        out += bytes(sbuf[:k])
    if dictionary is not None:
        n_sym, h16 = dictionary
        db = (C.c_uint8 * 32)()
        k = lib.cz_container_write_dictionary(db, len(db), int(n_sym), (C.c_uint8 * 16)(*h16))
        assert k, "dictionary section write failed"
        out += bytes(db[:k])
    if match_order:
        mb = (C.c_uint8 * 16)()
        k = lib.cz_container_write_match(mb, len(mb), int(match_order))
        assert k, "match section write failed"
        out += bytes(mb[:k])
    for p in payloads:
        out += p
    return bytes(out)


def read_container(blob: bytes):
    """Returns (fields dict, repr bytes, gates list or None, engine, seg_tokens, payload list).  A container with CZ_FLAG_DICTIONARY
    has fields["dictionary"] = (n_symbols, BLAKE3-128 of the symbols), as dictionary_id() gives them; one with CZ_FLAG_MATCH has
    fields["match_order"], the order of its MAT1 section."""
    buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
    h = _lib.HeaderV2()
    ro = C.c_size_t()
    n = lib.cz_container_read_header(buf, len(blob), C.byref(h), C.byref(ro))
    if not n:
        raise ValueError("bad container header")
    fields = {k: getattr(h, k) for k, _ in _lib.HeaderV2._fields_}
    for k in ("model_hash16", "tokenizer_hash16", "orig_hash16"):
        fields[k] = bytes(fields[k])
    rep = blob[ro.value : ro.value + h.model_file_repr_len]
    gates = None
    if h.reserved_flags & (1 << 2):
        rec = (C.c_uint8 * (len(blob)))()
        cnt = C.c_size_t()
        sub = (C.c_uint8 * (len(blob) - n)).from_buffer_copy(blob[n:])
        k = lib.cz_container_read_gates(sub, len(blob) - n, rec, len(blob), C.byref(cnt))
        if not k:
            raise ValueError("invalid gating magic")
        gates = list(rec[: cnt.value])
        n += k
    engine, seg_tokens = 0, None
    if h.reserved_flags & CZ_FLAG_SEGMENTS:
        sub = (C.c_uint8 * (len(blob) - n)).from_buffer_copy(blob[n:])
        cnt = C.c_size_t()
        eng = C.c_int()
        k = lib.cz_container_read_segments(sub, len(blob) - n, C.byref(eng), None, None, 0, C.byref(cnt))
        if not k:
            raise ValueError("bad segment table")
        st = np.zeros(cnt.value, np.uint64)
        sb = np.zeros(cnt.value, np.uint64)
        lib.cz_container_read_segments(sub, len(blob) - n, C.byref(eng), st.ctypes.data_as(_lib.u64p), sb.ctypes.data_as(_lib.u64p), cnt.value,
                                       C.byref(cnt))
        n += k
        engine, seg_tokens = eng.value, st
        n = _read_match(blob, _read_dictionary(blob, n, h, fields), h, fields)
        if int(sb.sum()) != len(blob) - n:
            raise ValueError(f"segment table declares {int(sb.sum())} payload bytes but {len(blob) - n} follow it")
        if int(st.sum()) != int(h.token_count):
            raise ValueError("segment table does not add up to token_count")
        payloads = []
        for b in sb:
            payloads.append(blob[n : n + int(b)])
            n += int(b)
    else:
        n = _read_match(blob, _read_dictionary(blob, n, h, fields), h, fields)
        payloads = [blob[n:]]
    return fields, rep, gates, engine, seg_tokens, payloads


def _read_dictionary(blob, n, h, fields):
    """the DIC1 section at blob[n:] when the header has CZ_FLAG_DICTIONARY: fills fields["dictionary"], returns the offset after it"""
    if not h.reserved_flags & CZ_FLAG_DICTIONARY:
        return n
    if h.reserved_flags & _lib.CZ_FLAG_STORED:
        raise ValueError("DICTIONARY marks a coded payload: invalid with STORED")
    sub = (C.c_uint8 * max(1, len(blob) - n)).from_buffer_copy(blob[n:] or b"\0")
    cnt = C.c_uint64()
    h16 = (C.c_uint8 * 16)()
    k = lib.cz_container_read_dictionary(sub, len(blob) - n, C.byref(cnt), h16)
    if not k:
        raise ValueError("bad dictionary section")
    fields["dictionary"] = (int(cnt.value), bytes(h16))
    return n + k


def _read_match(blob, n, h, fields):
    """the MAT1 section at blob[n:] when the header has CZ_FLAG_MATCH: fills fields["match_order"], returns the offset after it.  A flag
    without its section, a truncated section or an order outside [1, 16] raises ValueError."""
    if not h.reserved_flags & CZ_FLAG_MATCH:
        return n
    if h.reserved_flags & _lib.CZ_FLAG_STORED:
        raise ValueError("MATCH marks a coded payload: invalid with STORED")
    sub = (C.c_uint8 * max(1, len(blob) - n)).from_buffer_copy(blob[n:] or b"\0")
    order = C.c_uint32()
    k = lib.cz_container_read_match(sub, len(blob) - n, C.byref(order))
    if not k:
        raise ValueError("bad match section")
    fields["match_order"] = int(order.value)
    return n + k
