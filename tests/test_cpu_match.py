"""Match model without a GPU: hand-derived answers of the rule (tests/match_ref.py), the MAT1 container section in C and Python, the STORED
exclusion, decode waves keyed by the order, and the CLI's refusals."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import match_ref  # noqa: E402
from candlezip_b200 import _lib, codec, container  # noqa: E402
from candlezip_b200.__main__ import main  # noqa: E402

N = match_ref.NONE


def test_match_known_answers_k1():
    # i = 3: context (5) last seen before position 1, one symbol of agreement -> bucket 0, W from no history = 1/2
    # i = 4: context (6) before position 2, two symbols agree (6, 5) -> bucket 1, its own counts start at zero
    pred, w, b = match_ref.segment_predictions([5, 6, 5, 6, 5], 1)
    assert pred == [N, N, N, 6, 5] and w == [0, 0, 0, 1 << 29, 1 << 29] and b == [-1, -1, -1, 0, 1]
    # i = 3 misses in bucket 0 (predicts 1, sees 2); i = 5 is bucket 0 again with 0 hits of 1 try: p16 = (1 << 16) // 4, W = 2^28
    pred, w, b = match_ref.segment_predictions([9, 1, 9, 2, 9, 1], 1)
    assert pred == [N, N, N, 1, N, 2] and w == [0, 0, 0, 1 << 29, 0, 1 << 28] and b == [-1, -1, -1, 0, -1, 0]


def test_match_hash_collision_gives_no_prediction():
    assert match_ref.context_key([0]) == match_ref.context_key([709804])  # two one-symbol contexts with the same 18-bit key
    pred, w, _ = match_ref.segment_predictions([0, 3, 709804, 4, 0, 5], 1)
    assert pred == [N] * 6 and w == [0] * 6  # verify finds len 0 < K at both collisions
    pred, _, _ = match_ref.segment_predictions([0, 3, 0, 4], 1)  # without the collision position 3 is predicted
    assert pred == [N, N, N, 3]


@pytest.mark.parametrize("K", [1, 4, 16])
def test_match_length_capped(K):
    period = list(range(100, 100 + K + 1))  # no K-symbol context repeats inside one period
    t = period * (4 + (K + match_ref.NB) // len(period))  # long enough for the run to reach the cap
    pred, w, b = match_ref.segment_predictions(t, K)
    p = len(period)
    for i in range(len(t)):
        if i < p + K:  # the context of position i first repeats at i = p + K (seen before position K)
            assert pred[i] == N, i
        else:  # j = i - p; the contexts agree back to the segment's start or to the cap
            assert pred[i] == t[i] and b[i] == min(i - p, K + match_ref.NB - 1) - K, i
    assert max(b) == match_ref.NB - 1  # len reaches K + 15 and stops there
    last = max(i for i in range(len(t)) if b[i] == match_ref.NB - 1)
    tries = sum(1 for i in range(last) if b[i] == match_ref.NB - 1)
    assert w[last] == match_ref.weight(tries, tries)  # every earlier prediction of the top bucket was right


def test_match_counts_reset_per_segment():
    seg = [9, 1, 9, 2, 9, 1]
    pred, w = match_ref.predictions(seg + seg, np.array([0, 6, 12], np.uint64), 1)
    one = match_ref.segment_predictions(seg, 1)
    assert list(pred[:6]) == one[0] and list(pred[6:]) == one[0] and list(w[6:]) == one[1]
    whole, _ = match_ref.predictions(seg + seg, np.array([0, 12], np.uint64), 1)
    assert list(whole[6:]) != one[0]  # as one segment the history carries over


def test_match_interval_list():
    ids = [5, 6, 5, 6, 7]
    pred, w, _ = match_ref.segment_predictions(ids, 1)
    lo, hi = [10, 20, 30, 40, 50], [11, 21, 31, 41, 51]
    lst = match_ref.interval_list(ids, pred, w, lo, hi)
    # 3 tokens without a prediction, a hit (flag only), a miss (flag, then the model's interval)
    assert lst == [(10, 11), (20, 21), (30, 31), (0, 1 << 29), (1 << 29, 1 << 30), (50, 51)]


# ---- container ----------------------------------------------------------------------------------------------------------------------

def _fields(flags=0):
    return dict(token_count=3, orig_len_bytes=3, vocab_size=256, reserved_flags=flags)


def test_mat1_c_writer_reader():
    buf = (C.c_uint8 * 16)()
    for k in (1, 7, 16):
        n = _lib.lib.cz_container_write_match(buf, 16, k)
        assert n == 5 and bytes(buf[:5]) == b"MAT1" + bytes([k])
        o = C.c_uint32()
        assert _lib.lib.cz_container_read_match(buf, n, C.byref(o)) == 5 and o.value == k
    for k in (0, 17, 300):
        assert _lib.lib.cz_container_write_match(buf, 16, k) == 0
    assert _lib.lib.cz_container_write_match(buf, 4, 3) == 0  # no room
    o = C.c_uint32()
    for bad in (b"MAT1", b"MAT1\x00", b"MAT1\x11", b"MAT1\x80", b"MAT1\xac\x02", b"MATX\x04", b"MAT"):
        src = (C.c_uint8 * max(1, len(bad))).from_buffer_copy(bad or b"\0")
        assert _lib.lib.cz_container_read_match(src, len(bad), C.byref(o)) == 0, bad


@pytest.mark.parametrize("seg_tokens", [None, [2, 1]])
@pytest.mark.parametrize("dictionary", [None, (5, b"\1" * 16)])
def test_mat1_python_round_trip(seg_tokens, dictionary):
    pays = [b"\x40\x41", b"\x42"] if seg_tokens else [b"\x40\x41\x42"]
    blob = container.write_container(_fields(_lib.CZ_FLAG_PDF_FLOOR), b"m", pays, seg_tokens=seg_tokens, dictionary=dictionary, match_order=4)
    f, _, _, _, st, got = container.read_container(blob)
    assert f["match_order"] == 4 and f["reserved_flags"] & _lib.CZ_FLAG_MATCH and f["reserved_flags"] & _lib.CZ_FLAG_PDF_FLOOR
    assert got == pays and f.get("dictionary") == dictionary
    assert blob.index(b"MAT1") == len(blob) - sum(map(len, pays)) - 5  # right before the payloads, after DIC1
    plain = container.write_container(_fields(), b"m", pays, seg_tokens=seg_tokens, dictionary=dictionary)
    assert "match_order" not in container.read_container(plain)[0] and b"MAT1" not in plain


def test_mat1_reader_rejects_malformed():
    blob = container.write_container(_fields(), b"m", [b"\x40"], match_order=3)
    i = blob.index(b"MAT1")
    for bad in (blob[:i] + b"MAT1\x00" + blob[i + 5:], blob[:i] + b"MAT1\x11" + blob[i + 5:], blob[:i] + b"MAT1",
                blob[:i] + b"XXXX" + blob[i + 4:], blob[:i]):
        with pytest.raises(ValueError):
            container.read_container(bad)
    # the flag without its section
    plain = container.write_container(_fields(_lib.CZ_FLAG_MATCH), b"m", [b"\x40"])
    with pytest.raises(ValueError):
        container.read_container(plain)
    with pytest.raises(ValueError):
        container.write_container(_fields(), b"m", [b"\x40"], match_order=17)


def test_mat1_never_with_stored():
    with pytest.raises(ValueError):
        container.write_container(_fields(_lib.CZ_FLAG_STORED), b"m", [b"abc"], match_order=4)
    # a STORED payload that happens to start with MAT1 is just bytes; a STORED header that claims the flag is refused
    blob = container.write_container(_fields(_lib.CZ_FLAG_STORED), b"m", [b"MAT1\x04abc"])
    assert "match_order" not in container.read_container(blob)[0]
    forged = container.write_container(_fields(_lib.CZ_FLAG_STORED), b"m", [b"abc"])
    h = _lib.HeaderV2()
    ro = C.c_size_t()
    buf = (C.c_uint8 * len(forged)).from_buffer_copy(forged)
    n = _lib.lib.cz_container_read_header(buf, len(forged), C.byref(h), C.byref(ro))
    h.reserved_flags |= _lib.CZ_FLAG_MATCH
    out = (C.c_uint8 * (n + 64))()
    k = _lib.lib.cz_container_write_header(out, n + 64, C.byref(h), (C.c_uint8 * 1).from_buffer_copy(b"m"))
    with pytest.raises(ValueError, match="STORED"):
        container.read_container(bytes(out[:k]) + b"MAT1\x04abc")


def test_stored_fallback_writes_no_match_section():
    class ZeroWidthModel:
        cfg = dict(vocab=256, arch=0)
        engine = 0

        def encode(self, ids, **kw):
            assert kw.get("match_order") == 4
            raise _lib.CzError(_lib.CZ_ERR_ZERO_WIDTH, "zero width")

    blob = codec.compress(ZeroWidthModel(), b"abcabc", match_order=4)
    f = container.read_container(blob)[0]
    assert f["reserved_flags"] & _lib.CZ_FLAG_STORED and not f["reserved_flags"] & _lib.CZ_FLAG_MATCH and "match_order" not in f


def test_compress_rejects_bad_order():
    for bad in (-1, 17, 2.5, "4"):
        with pytest.raises(ValueError):
            codec.compress(None, b"abc", match_order=bad)
        with pytest.raises(ValueError):
            codec.compress_many(None, [b"abc"], match_order=bad)


def test_decode_waves_keyed_by_order():
    class M:
        cfg = dict(vocab=256, arch=0)
        engine = 0

    blobs = [codec.coded_container(M(), codec.header_fields(M(), b"abcd", 4, 0, 512, 512, b"\0" * 16, b"\0" * 16), b"m", [b"\x40"],
                                   np.array([0, 4], np.uint64), None, k) for k in (0, 4, 4, 7)]
    keys = [codec._parse(M(), b, verify=False).key for b in blobs]
    assert [k[5] for k in keys] == [0, 4, 4, 7] and keys[0][:5] == keys[1][:5] == keys[3][:5]
    waves = codec.decode_waves([(k, [4]) for k in keys], 100)
    assert sorted(sorted(f for f, _, _ in items) for _, items in waves) == [[0], [1, 2], [3]]


@pytest.mark.parametrize("argv", [
    ["analyze", "x", "--match-order", "4"],
    ["decompress", "x", "--match-order", "4"],
    ["decompress-many", "x", "--match-order", "4"],
    ["compress", "x", "--match-order", "4", "--reuse-scan-dir", "d"],
    ["self-test", "x", "--match-order", "4", "--reuse-scan-dir", "d"],
    ["compress", "x", "--match-order", "0"],
    ["compress", "x", "--match-order", "17"],
])
def test_cli_refuses_match_order(argv, capsys):
    with pytest.raises(SystemExit) as e:
        main(argv)
    assert e.value.code == 2
    assert "--match-order" in capsys.readouterr().err
