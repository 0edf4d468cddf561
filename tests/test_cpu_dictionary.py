"""CPU suite for preset dictionaries: the prefix-aware chunk schedule (cz_schedule_chunks_prefixed) against the plain schedule of
dictionary ++ tokens, the DIC1 container section and its refusals, the file-level checks that refuse a missing or different dictionary
before any decode call (with a fake model), and the CLI's refusals."""
import numpy as np
import pytest

from candlezip_b200 import _lib, codec, container, split_segments


def _chunks(n, context, reprime, n_prefix=None):
    f = _lib.lib.cz_schedule_chunks if n_prefix is None else _lib.lib.cz_schedule_chunks_prefixed
    args = (int(n), int(context), int(reprime)) if n_prefix is None else (int(n), int(n_prefix), int(context), int(reprime))
    k = int(f(*args, None, None, None, None, 0))
    first, n_coded = np.zeros(max(k, 1), np.uint64), np.zeros(max(k, 1), np.uint32)
    ps, pl = np.zeros(max(k, 1), np.uint64), np.zeros(max(k, 1), np.uint32)
    assert f(*args, first.ctypes.data_as(_lib.u64p), n_coded.ctypes.data_as(_lib.u32p), ps.ctypes.data_as(_lib.u64p),
             pl.ctypes.data_as(_lib.u32p), k) == k
    return [tuple(int(x) for x in t) for t in zip(first[:k], n_coded[:k], ps[:k], pl[:k])]


def _clipped(n, d, context, reprime):
    """cz_schedule_chunks(d + n) clipped to coded indices >= d, the clipped positions moved into the prime"""
    out = []
    for first, k, ps, pl in _chunks(d + n, context, reprime):
        if first + k <= d:
            continue
        skip = max(0, d - first)
        out.append((first + skip - d, k - skip, ps, pl + skip))
    return out


@pytest.mark.parametrize("reprime", [1, 7, 512])
@pytest.mark.parametrize("d", [1, 510, 511, 512, 513, 1500, 5000])
def test_prefixed_schedule_is_the_clipped_plain_schedule(d, reprime):
    for n in (0, 1, 2, 7, 300, 511, 512, 513, 1400):
        for context in (512, 100):
            got = _chunks(n, context, reprime, d)
            assert got == _clipped(n, d, context, reprime), (d, reprime, n, context)
            assert sum(k for _, k, _, _ in got) == n
            if not n:
                continue
            # the first chunk's prime is BOS and dictionary positions only, and it ends right before the first coded token
            first, k, ps, pl = got[0]
            assert first == 0 and ps + pl == 1 + d
            # row bound: a chunk has the rows its unclipped twin has, so at most one reprime chunk of extra prime rows
            eff = min(context, 511)
            for f, k, ps, pl in got:
                assert pl + k - 1 <= eff + max(reprime, eff) - 1, (d, reprime, n, context, f, k, pl)
                assert pl <= eff + max(reprime, eff) - 1
    # no prefix: the plain schedule
    assert _chunks(777, 512, 512, 0) == _chunks(777, 512, 512)


def test_prefixed_schedule_default_first_chunk_rows():
    """at --context 512 / --reprime-interval 512 the first run chunk primes with at most 1,022 positions"""
    worst = max(_chunks(10, 512, 512, d)[0][3] for d in range(1, 3000))
    assert worst == 1022


def _fields(n_tokens, flags=0):
    return dict(bos_token_id=0, token_count=n_tokens, orig_len_bytes=n_tokens, vocab_size=256, reserved_flags=flags)


def test_dic1_round_trip():
    dic = container.dictionary_id(np.arange(37, dtype=np.uint32))
    assert dic[0] == 37 and len(dic[1]) == 16
    assert dic != container.dictionary_id(np.arange(1, 38, dtype=np.uint32))
    assert container.dictionary_id([258]) == (1, container.blake3_16((258).to_bytes(4, "little")))
    pays = [b"abc", b"", b"defgh"]
    for flags in (0, _lib.CZ_FLAG_PDF_FLOOR):
        one = container.write_container(_fields(9, flags), b"m", [b"xyz"], dictionary=dic)
        f, rep, gates, _, seg, got = container.read_container(one)
        assert f["dictionary"] == dic and f["reserved_flags"] == flags | _lib.CZ_FLAG_DICTIONARY and got == [b"xyz"] and seg is None
        plain = container.write_container(_fields(9, flags), b"m", [b"xyz"])
        assert "dictionary" not in container.read_container(plain)[0]
        assert len(one) == len(plain) + 4 + 1 + 16
        segd = container.write_container(_fields(9, flags), b"m", pays, seg_tokens=[3, 0, 6], dictionary=dic)
        f, _, _, _, seg, got = container.read_container(segd)
        assert f["dictionary"] == dic and list(seg) == [3, 0, 6] and got == pays
        assert f["reserved_flags"] == flags | _lib.CZ_FLAG_DICTIONARY | _lib.CZ_FLAG_SEGMENTS
    # the C section on its own
    buf = (np.zeros(64, np.uint8))
    h = (b"\x11" * 16)
    for n in (1, 127, 128, 2 ** 40):
        k = _lib.lib.cz_container_write_dictionary(buf.ctypes.data_as(_lib.u8p), 64, n, np.frombuffer(h, np.uint8).ctypes.data_as(_lib.u8p))
        assert k == 4 + len(_varint(n)) + 16 and bytes(buf[:4]) == b"DIC1"
        cnt, h16 = np.zeros(1, np.uint64), np.zeros(16, np.uint8)
        assert _lib.lib.cz_container_read_dictionary(buf.ctypes.data_as(_lib.u8p), k, cnt.ctypes.data_as(_lib.u64p),
                                                     h16.ctypes.data_as(_lib.u8p)) == k
        assert int(cnt[0]) == n and h16.tobytes() == h
    assert _lib.lib.cz_container_write_dictionary(buf.ctypes.data_as(_lib.u8p), 20, 1, buf.ctypes.data_as(_lib.u8p)) == 0


def _varint(v):
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def _read_dic(b):
    a = np.frombuffer(b + b"\0", np.uint8).copy()
    cnt, h16 = np.zeros(1, np.uint64), np.zeros(16, np.uint8)
    return int(_lib.lib.cz_container_read_dictionary(a.ctypes.data_as(_lib.u8p), len(b), cnt.ctypes.data_as(_lib.u64p),
                                                     h16.ctypes.data_as(_lib.u8p)))


def test_dic1_refusals():
    good = b"DIC1" + _varint(300) + b"\x22" * 16
    assert _read_dic(good) == len(good)
    for k in range(len(good)):  # every truncation, including one inside the varint
        assert _read_dic(good[:k]) == 0, k
    assert _read_dic(b"DIC2" + good[4:]) == 0
    assert _read_dic(b"DIC1" + _varint(0) + b"\x22" * 16) == 0  # an empty dictionary is never written
    assert _read_dic(b"DIC1" + b"\xff" * 11 + b"\x22" * 16) == 0  # a count that does not end (or overflows 64 bits)
    assert _read_dic(b"DIC1" + b"\x80" * 3) == 0  # a count running past the buffer
    dic = container.dictionary_id([1, 2, 3])
    blob = container.write_container(_fields(4), b"m", [b"payload"], dictionary=dic)
    cut = blob.index(b"DIC1")
    with pytest.raises(ValueError, match="bad dictionary section"):
        container.read_container(blob[: cut + 10])
    with pytest.raises(ValueError, match="bad dictionary section"):
        container.read_container(blob[:cut] + b"XXXX" + blob[cut + 4 :])
    segd = container.write_container(_fields(4), b"m", [b"ab", b"cd"], seg_tokens=[2, 2], dictionary=dic)
    with pytest.raises(ValueError):
        container.read_container(segd[:-1])  # the segment table still accounts for every payload byte after the section
    # STORED and DICTIONARY never go together
    with pytest.raises(ValueError, match="STORED"):
        container.write_container(_fields(4, _lib.CZ_FLAG_STORED), b"m", [b"abcd"], dictionary=dic)
    both = container.write_container(_fields(4, _lib.CZ_FLAG_STORED | _lib.CZ_FLAG_DICTIONARY), b"m", [good + b"abcd"])
    with pytest.raises(ValueError, match="STORED"):
        container.read_container(both)


class DictFakeModel:
    """Model.encode / Model.decode stand-in whose payload records the dictionary it was coded with: b"P", the dictionary's BLAKE3-128 or
    16 zero bytes, then the ids.  Records every call."""

    def __init__(self):
        self.cfg = dict(arch=0, vocab=256)
        self.engine = 0
        self.encodes, self.decodes = [], []

    @staticmethod
    def _tag(dictionary):
        return b"\0" * 16 if dictionary is None else container.dictionary_id(dictionary)[1]

    def encode(self, ids, n_segments=1, bos=0, context=512, reprime_interval=512, seg_start=None, pdf_floor=False, zero_width_out=False,
               dictionary=None):
        ids = np.asarray(ids, np.uint32)
        seg = split_segments(len(ids), n_segments) if seg_start is None else np.asarray(seg_start, np.uint64)
        self.encodes.append(dict(n_tokens=len(ids), dictionary=None if dictionary is None else [int(x) for x in dictionary]))
        pays = [b"P" + self._tag(dictionary) + ids[int(seg[g]) : int(seg[g + 1])].tobytes() for g in range(len(seg) - 1)]
        zw = np.full(len(seg) - 1, _lib.NO_ZERO_WIDTH, np.uint64)
        return (pays, seg, zw) if zero_width_out else (pays, seg)

    def decode(self, payloads, seg_start, bos=0, context=512, reprime_interval=512, pdf_floor=False, dictionary=None):
        lens = np.diff(np.asarray(seg_start, np.uint64))
        self.decodes.append(dict(n_segments=len(payloads), dictionary=None if dictionary is None else [int(x) for x in dictionary]))
        out = []
        for p, n in zip(payloads, lens):
            assert p[:17] == b"P" + self._tag(dictionary)
            out.append(np.frombuffer(p[17:], np.uint32))
        return np.concatenate(out).astype(np.uint32) if out else np.zeros(0, np.uint32)


def test_dictionary_round_trips_and_empty_writes_todays_container():
    m = DictFakeModel()
    data, dic = b"hello dictionary world", b"hello "
    blob = codec.compress(m, data, n_segments=2, dictionary=dic)
    f = container.read_container(blob)[0]
    assert f["dictionary"] == container.dictionary_id(np.frombuffer(dic, np.uint8).astype(np.uint32))
    assert m.encodes[-1]["dictionary"] == list(dic)
    assert codec.decompress(m, blob, dictionary=dic) == data and m.decodes[-1]["dictionary"] == list(dic)
    plain = codec.compress(m, data, n_segments=2)
    assert codec.compress(m, data, n_segments=2, dictionary=b"") == plain and codec.compress(m, data, n_segments=2, dictionary=None) == plain
    assert m.encodes[-1]["dictionary"] is None
    # a container without a dictionary decodes without one, whatever is offered
    m.decodes.clear()
    assert codec.decompress(m, plain, dictionary=dic) == data and m.decodes == [dict(n_segments=2, dictionary=None)]


def test_missing_or_different_dictionary_raises_before_any_decode():
    m = DictFakeModel()
    datas = [b"alpha beta", b"gamma", b"", b"delta epsilon"]
    dic = b"beta gamma"
    blobs = codec.compress_many(m, datas, n_segments=2, dictionary=dic)
    assert len(m.encodes) == 1 and m.encodes[0]["dictionary"] == list(dic)
    assert blobs == [codec.compress(m, d, n_segments=2, dictionary=dic) for d in datas]
    m.decodes.clear()
    with pytest.raises(ValueError, match="none was given"):
        codec.decompress(m, blobs[0])
    with pytest.raises(ValueError, match="different dictionary"):
        codec.decompress(m, blobs[0], dictionary=b"beta gammA")
    with pytest.raises(ValueError, match=r"^blob 0: .*none was given"):
        codec.decompress_many(m, blobs)
    plain = codec.compress(m, b"zeta", n_segments=1)
    with pytest.raises(ValueError, match=r"^blob 2: .*different dictionary"):
        codec.decompress_many(m, [plain, blobs[1], codec.compress(m, b"eta", dictionary=b"other")], dictionary=dic)
    assert m.decodes == []
    # mixed containers: with and without the dictionary never share a call
    assert codec.decompress_many(m, blobs + [plain], dictionary=dic) == datas + [b"zeta"]
    assert sorted(str(c["dictionary"]) for c in m.decodes) == sorted([str(list(dic)), "None"])


def test_decode_keys_carry_the_dictionary_hash():
    m = DictFakeModel()
    a = codec._parse(m, codec.compress(m, b"abc", dictionary=b"x"), True, np.array([120], np.uint32))
    b = codec._parse(m, codec.compress(m, b"abc"), True)
    assert a.key[:4] == b.key[:4] and a.key[4] == container.dictionary_id([120])[1] and b.key[4] is None


def test_cli_refuses_dictionary_with_the_gate_replay(capsys):
    from candlezip_b200.__main__ import main

    for argv in (["compress", "a", "--dictionary", "d", "--reuse-scan-dir", "s"], ["decompress", "a", "--dictionary", "d", "--reuse-scan-dir", "s"],
                 ["self-test", "a", "--dictionary", "d", "--reuse-scan-dir", "s"]):
        with pytest.raises(SystemExit) as e:
            main(argv)
        assert e.value.code == 2, argv
    assert "--dictionary is not available with --reuse-scan-dir" in capsys.readouterr().err


def test_model_refuses_bad_dictionaries_without_a_device():
    """cz_model_set_dictionary validates and copies on the host: a model on a device-less context takes it"""
    import candlezip_b200 as cz

    ctx = cz.Context(-1)
    m = cz.Model(ctx, cz.SMOLLM_TINY)
    m.set_dictionary(np.arange(1024, dtype=np.uint32))
    m.set_dictionary(None)
    m.set_dictionary([])
    with pytest.raises(cz.CzError) as e:
        m.set_dictionary([5, 1024, 7])
    assert e.value.code == _lib.CZ_ERR_SYMBOL_RANGE and "at index 1" in str(e.value)
    assert _lib.lib.cz_model_set_dictionary(m._h, None, 3) == _lib.CZ_ERR_INVALID
    r = cz.Model(ctx, dict(cz.RWKV7_0P1B, vocab=512))
    r.set_dictionary([511, 512, 767])  # literal escapes are in the RWKV-7 coded alphabet
    with pytest.raises(cz.CzError) as e:
        r.set_dictionary([768])
    assert e.value.code == _lib.CZ_ERR_SYMBOL_RANGE
    m.close()
    r.close()
    ctx.close()
