"""CPU suite for per-token code lengths (codec.analyze, Model.analyze, `python -m candlezip_b200 analyze`): the summary and its position
buckets on hand-made arrays, the segment / chunk position arrays against cz_schedule_chunks, the CLI's flag refusals and the argument
checks that come before any device work."""
import json

import numpy as np
import pytest

import candlezip_b200 as cz
from candlezip_b200 import _lib, codec
from candlezip_b200.__main__ import main
from candlezip_b200.api import code_length_bits, split_segments


def test_code_length_bits():
    lo = np.array([0, 0, 5, 1 << 29, 7], np.uint32)
    hi = np.array([1 << 30, 1, 6, 1 << 30, 7], np.uint32)
    b = code_length_bits(lo, hi)
    assert b[0] == 0.0 and b[1] == 30.0 and b[2] == 30.0 and b[3] == 1.0 and b[4] == np.inf


def test_pos_bucket_and_labels():
    pos = np.arange(0, 70)
    bk = codec.pos_bucket(pos)
    want = [0 if p == 0 else int(p).bit_length() for p in pos]
    assert bk.tolist() == want
    assert [codec.bucket_label(b) for b in range(5)] == ["0", "1", "2-3", "4-7", "8-15"]
    assert codec.pos_bucket([1 << 40, (1 << 40) - 1]).tolist() == [41, 40]


def test_summary_on_hand_made_arrays():
    bits = np.array([1.0, 2.0, np.inf, 4.0, 0.5, np.inf, 3.0])
    ent = np.array([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 3.5])
    seg = np.array([0, 0, 0, 0, 1, 1, 1])
    spos = np.array([0, 1, 2, 3, 0, 1, 2])
    cpos = np.array([0, 1, 0, 1, 0, 1, 2])
    s = codec.summarize(bits, ent, seg, spos, cpos, [3, 2], 10)
    assert s["tokens"] == 7 and s["bytes"] == 10
    assert s["bits"] == 10.5 and s["bits_per_byte"] == 1.05
    assert s["payload_bits"] == 40 and s["payload_bits_per_byte"] == 4.0
    assert s["mean_bits"] == 10.5 / 5 and s["mean_entropy"] == ent.mean()
    assert s["zero_width"] == 2 and s["first_zero_width"] == [2, 5]
    assert s["segments"] == [dict(tokens=4, bits=7.0, zero_width=1, payload_bits=24, entropy=5.0),
                             dict(tokens=3, bits=3.5, zero_width=1, payload_bits=16, entropy=9.0)]
    by_c = {b["bucket"]: b for b in s["by_chunk_position"]}
    assert set(by_c) == {"0", "1", "2-3"}
    assert by_c["0"]["tokens"] == 3 and by_c["0"]["zero_width"] == 1 and by_c["0"]["mean_bits"] == 0.75
    assert by_c["0"]["mean_entropy"] == (0.5 + 1.5 + 2.5) / 3
    assert by_c["1"]["tokens"] == 3 and by_c["1"]["zero_width"] == 1 and by_c["1"]["mean_bits"] == 3.0
    assert by_c["2-3"] == dict(bucket="2-3", tokens=1, zero_width=0, mean_bits=3.0, mean_entropy=3.5)
    by_s = {b["bucket"]: b for b in s["by_segment_position"]}
    assert by_s["2-3"]["tokens"] == 3 and by_s["2-3"]["mean_bits"] == 3.5 and by_s["2-3"]["zero_width"] == 1
    # the bucket totals add up to the whole
    for key in ("by_chunk_position", "by_segment_position"):
        assert sum(b["tokens"] for b in s[key]) == 7 and sum(b["zero_width"] for b in s[key]) == 2
    json.dumps(s)  # (the CLI stores it as JSON)


def test_summary_edge_cases():
    s = codec.summarize(np.zeros(0), np.zeros(0), np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64), [1], 0)
    assert s["tokens"] == 0 and s["bits_per_byte"] is None and s["mean_bits"] is None and s["mean_entropy"] is None
    assert s["by_chunk_position"] == [] and s["segments"][0]["payload_bits"] == 8
    s = codec.summarize(np.array([np.inf]), np.array([2.0]), [0], [0], [0], [4], 1)
    assert s["bits"] == 0.0 and s["mean_bits"] is None and s["zero_width"] == 1 and s["by_chunk_position"][0]["mean_bits"] is None


@pytest.mark.parametrize("reprime_interval", [1, 7, 100, 512, 777])
@pytest.mark.parametrize("n,n_segments", [(0, 1), (1, 1), (511, 1), (1300, 1), (2600, 3), (5000, 7)])
def test_positions_against_cz_schedule_chunks(n, n_segments, reprime_interval):
    seg_start = split_segments(n, n_segments)
    seg, pos, chunk, cpos = codec.token_positions(seg_start, 512, reprime_interval)
    assert seg.shape == pos.shape == chunk.shape == cpos.shape == (n,)
    for g in range(len(seg_start) - 1):
        a, b = int(seg_start[g]), int(seg_start[g + 1])
        assert np.all(seg[a:b] == g) and np.array_equal(pos[a:b], np.arange(b - a))
        cap = 1 << 14
        first, ncod = np.zeros(cap, np.uint64), np.zeros(cap, np.uint32)
        k = _lib.lib.cz_schedule_chunks(b - a, 512, reprime_interval, first.ctypes.data_as(_lib.u64p), ncod.ctypes.data_as(_lib.u32p), None,
                                        None, cap)
        assert sum(int(x) for x in ncod[:k]) == b - a
        for c in range(k):
            f, m = a + int(first[c]), int(ncod[c])
            assert np.all(chunk[f:f + m] == c) and np.array_equal(cpos[f:f + m], np.arange(m)), (g, c)
        # a reprime happens every reprime_interval tokens once the context is full (511 tokens of history)
        if b - a > 0:
            starts = np.nonzero(cpos[a:b] == 0)[0]
            assert starts[0] == 0
            assert all(s % reprime_interval == 0 and s >= 510 for s in starts[1:])
    # one chunk per segment without reprimes (RWKV-7)
    seg2, pos2, chunk2, cpos2 = codec.token_positions(seg_start, 512, reprime_interval, reprime=False)
    assert np.array_equal(seg2, seg) and np.array_equal(pos2, pos) and not chunk2.any() and np.array_equal(cpos2, pos)


@pytest.mark.parametrize("argv,msg", [
    (["compress", "x", "--pdf-floor"], "--pdf-floor"),
    (["self-test", "x", "--pdf-floor"], "--pdf-floor"),
    (["decompress", "x", "--pdf-floor"], "--pdf-floor"),
    (["compress-many", "x", "--pdf-floor"], "--pdf-floor"),
    (["analyze", "x", "--pdf-floor", "--backend", "rwkv7"], "--pdf-floor"),
    (["analyze", "x", "--reuse-scan-dir", "d"], "--reuse-scan-dir"),
    (["analyze", "x", "--on-zero-width", "floor"], "--on-zero-width"),
    (["analyze", "x", "--out-dir", "d"], "--out-dir"),
    (["analyze", "x", "--max-streams", "4"], "--max-streams"),
])
def test_cli_refusals(argv, msg, capsys):
    with pytest.raises(SystemExit) as e:
        main(argv)
    assert e.value.code == 2
    assert msg in capsys.readouterr().err


@pytest.fixture(scope="module")
def host_model():
    ctx = cz.Context(-1)  # host-only: the argument checks come before anything needs a device
    m = cz.Model(ctx, cz.SMOLLM_TINY)
    r = cz.Model(ctx, dict(cz.RWKV7_0P1B, vocab=1024, d_model=64, n_layers=1, n_heads=1, d_ffn=256))
    yield m, r
    m.close()
    r.close()
    ctx.close()


def test_model_analyze_argument_checks(host_model):
    m, r = host_model
    ids = np.arange(10, dtype=np.uint32)
    for kw in (dict(n_segments=0), dict(context=0), dict(reprime_interval=0), dict(seg_start=[0, 5]), dict(seg_start=[1, 10]),
               dict(seg_start=[0, 7, 3, 10]), dict(seg_start=[10])):
        with pytest.raises(ValueError):
            m.analyze(ids, **kw)
    with pytest.raises(ValueError):
        r.analyze(ids, pdf_floor=True)
    # valid arguments reach the encode call, which needs a device
    with pytest.raises(cz.CzError) as e:
        m.analyze(ids, n_segments=2)
    assert e.value.code == _lib.CZ_ERR_NO_DEVICE


def test_code_length_sink_arguments(host_model):
    m, _ = host_model
    lo = np.zeros(4, np.uint32)
    ent = np.zeros(4, np.float64)
    set_out = _lib.lib.cz_model_set_code_length_out
    assert set_out(m._h, lo.ctypes.data_as(_lib.u32p), None, None, 0) == _lib.CZ_ERR_INVALID
    assert set_out(m._h, None, None, ent.ctypes.data_as(_lib.f64p), 0) == _lib.CZ_ERR_INVALID
    assert set_out(None, None, None, None, 0) == _lib.CZ_ERR_INVALID
    assert set_out(m._h, lo.ctypes.data_as(_lib.u32p), None, ent.ctypes.data_as(_lib.f64p), 4) == _lib.CZ_OK
    assert set_out(m._h, None, None, None, 0) == _lib.CZ_OK
    # the K1 entry point needs a device
    ctx = cz.Context(-1)
    with pytest.raises(cz.CzError) as e:
        ctx.cdf_entropy(np.zeros((8, 2), np.float32))
    assert e.value.code == _lib.CZ_ERR_NO_DEVICE
    ctx.close()
