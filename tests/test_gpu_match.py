"""GPU suite for the match model (cz_model_set_match): per-token predictions and weights of encode and decode equal the sequential
restatement (tests/match_ref.py) on SmolLM (both engines) and RWKV-7 (literal escapes included); payloads are the oracle coder over the
interval list built on the host from those predictions and the match-off model intervals; round trips over segment splits, orders,
fixtures, the pdf floor, a dictionary and the many-file paths; the zero-width report and both fallbacks; the setting off changes
nothing; hint-prime events are refused; and the compression the rule gives on random-init SmolLM-135M."""
import os
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
from candlezip_b200 import _lib, codec, container
from test_gpu_dictionary import _rwkv_tiny
from test_gpu_pdf_floor import _greedy_with_one_surprise, _PairTokenizer, _peaky

import match_ref
import oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def _repetitive_ids(vocab, n, rng, literal_base=None):
    """text-like ids: phrases drawn from a small pool (many long repeats), some noise, RWKV-7 literal escapes when literal_base is set"""
    pool = [rng.integers(0, vocab, rng.integers(3, 40)).astype(np.uint32) for _ in range(12)]
    out = []
    while sum(map(len, out)) < n:
        out.append(pool[rng.integers(0, len(pool))] if rng.random() < 0.8 else rng.integers(0, vocab, rng.integers(1, 8)).astype(np.uint32))
    ids = np.concatenate(out)[:n].astype(np.uint32)
    if literal_base is not None:
        lit = rng.random(n) < 0.05
        ids[lit] = literal_base + (ids[lit] % 256)
    return ids


def _splits(n):
    """1 and 7 segments, and a ragged non-increasing split with a one-token and an empty segment"""
    ragged = [n // 2, n // 4, n - n // 2 - n // 4 - 1, 1, 0]
    ragged.sort(reverse=True)
    return [np.array([0, n], np.uint64), cz.split_segments(n, 7), np.concatenate([[0], np.cumsum(ragged)]).astype(np.uint64)]


def _check_call(gpu_ctx, model, ids, seg, K, **kw):
    """encode with the match model against the restatement and the oracle coder; decode back with the same predictions"""
    n = ids.shape[0]
    pred_e, w_e = model.watch_match(n)
    pays, _ = model.encode(ids, seg_start=seg, match_order=K, **kw)
    pred_e, w_e = pred_e.copy(), w_e.copy()
    want_pred, want_w = match_ref.predictions(ids, seg, K)
    assert np.array_equal(pred_e, want_pred), np.nonzero(pred_e != want_pred)[0][:5]
    assert np.array_equal(w_e, want_w), np.nonzero(w_e != want_w)[0][:5]
    # the model's intervals do not depend on the match model: a match-off run with the code-length sink gives them
    r = model.analyze(ids, seg_start=seg, pdf_floor=kw.get("pdf_floor", False), dictionary=kw.get("dictionary"))
    for g in range(len(seg) - 1):
        a, b = int(seg[g]), int(seg[g + 1])
        lst = match_ref.interval_list(ids[a:b], want_pred[a:b], want_w[a:b], r["c_lo"][a:b], r["c_hi"][a:b])
        assert oracle.ac_encode(lst) == pays[g], (g, K)
    pred_d, w_d = model.watch_match(n)
    out = model.decode(pays, seg, match_order=K, **kw)
    assert np.array_equal(out, ids)
    assert np.array_equal(pred_d, want_pred) and np.array_equal(w_d, want_w)
    model.watch_match(0)
    return pays, want_pred


def _run_backend(gpu_ctx, model, ids, **kw):
    for seg in _splits(ids.shape[0]):
        for K in (1, 4, 16):
            pays, pred = _check_call(gpu_ctx, model, ids, seg, K, **kw)
            assert np.any(pred != match_ref.NONE)
    # a segment coded alone (another wave, another packing) gets the same predictions and payload
    seg = cz.split_segments(ids.shape[0], 7)
    pays, _ = model.encode(ids, seg_start=seg, match_order=4, **kw)
    a, b = int(seg[3]), int(seg[4])
    pred, w = model.watch_match(b - a)
    alone, _ = model.encode(ids[a:b], match_order=4, **kw)
    want = match_ref.predictions(ids, seg, 4)
    assert alone[0] == pays[3] and np.array_equal(pred, want[0][a:b]) and np.array_equal(w, want[1][a:b])
    model.watch_match(0)


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_TCGEN05, _lib.CZ_ENGINE_SIMT])
def test_match_tiny_smollm(gpu_ctx, engine):
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(5, 0.05, 0.05)
    rng = np.random.default_rng(engine + 11)
    _run_backend(gpu_ctx, model, _repetitive_ids(cz.SMOLLM_TINY["vocab"], 1500, rng))
    model.close()


def test_match_tiny_rwkv7(gpu_ctx):
    model = _rwkv_tiny(gpu_ctx)
    rng = np.random.default_rng(3)
    v = int(model.cfg["vocab"])
    _run_backend(gpu_ctx, model, _repetitive_ids(v, 1200, rng, literal_base=v))
    model.close()


def test_match_tiny_floor_and_dictionary(gpu_ctx):
    """the pdf floor and a dictionary: the dictionary is not match history, and each setting combines with the match model"""
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
    rng = np.random.default_rng(9)
    ids = _repetitive_ids(1024, 1300, rng)
    dic = ids[:300].copy()  # the segment repeats the dictionary: still no prediction from it
    for seg in _splits(ids.shape[0])[:2]:
        _check_call(gpu_ctx, model, ids, seg, 4, pdf_floor=True)
        _check_call(gpu_ctx, model, ids, seg, 4, dictionary=dic)
    model.close()


def test_match_tiny_zero_width_and_fallbacks(gpu_ctx):
    """on a peaky model the zero-width report names the first NON-HIT token with an empty interval; both fallbacks round-trip"""
    model = _peaky(gpu_ctx)
    tok = _PairTokenizer()
    ids = _greedy_with_one_surprise(model, 1200, 700)
    seg = np.array([0, ids.shape[0]], np.uint64)
    r = model.analyze(ids)
    zw = np.nonzero(r["c_lo"] == r["c_hi"])[0]
    pred, _ = match_ref.predictions(ids, seg, 4)
    non_hit = [int(i) for i in zw if pred[i] != ids[i]]
    assert non_hit, "the test needs a zero-width token that the match model does not predict"
    _, _, first_zw = model.encode(ids, zero_width_out=True, match_order=4)
    assert int(first_zw[0]) == non_hit[0]
    with pytest.raises(cz.CzError) as e:
        model.encode(ids, match_order=4)
    assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH and f"coded index {non_hit[0]}:" in str(e.value)
    data = tok.decode_bytes(ids)
    for policy, flag in (("floor", _lib.CZ_FLAG_PDF_FLOOR), ("stored", _lib.CZ_FLAG_STORED)):
        blob = codec.compress(model, data, tok, on_zero_width=policy, match_order=4)
        f = container.read_container(blob)[0]
        assert f["reserved_flags"] & flag
        assert f.get("match_order") == (4 if policy == "floor" else None)
        assert codec.decompress(model, blob, tok) == data
        many = codec.compress_many(model, [data, data[:200]], tok, on_zero_width=policy, match_order=4)
        assert many[0] == blob and codec.decompress_many(model, many, tok) == [data, data[:200]]
    model.close()


def test_match_tiny_off_changes_nothing(gpu_ctx):
    """order 0 after an order-4 call launches what a model that never used the match model launches, and writes the same bytes"""
    rng = np.random.default_rng(4)
    ids = _repetitive_ids(1024, 1000, rng)
    runs = []
    for use in (False, True):
        model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
        if use:
            model.decode(*model.encode(ids, n_segments=3, match_order=4), match_order=4)
        l0 = gpu_ctx.launch_count()
        pays, seg = model.encode(ids, n_segments=3)
        l1 = gpu_ctx.launch_count()
        out = model.decode(pays, seg)
        l2 = gpu_ctx.launch_count()
        assert np.array_equal(out, ids)
        runs.append((pays, l1 - l0, l2 - l1))
        model.close()
    assert runs[0] == runs[1]


def test_match_events_unsupported(gpu_ctx):
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
    ids = np.arange(300, dtype=np.uint32) % 50
    ev = [(100, [1, 2, 3], 150)]
    with pytest.raises(cz.CzError) as e:
        model.encode(ids, events=ev, match_order=4)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    pays, seg = model.encode(ids, events=ev)
    with pytest.raises(cz.CzError) as e:
        model.decode(pays, seg, events=ev, match_order=4)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    with pytest.raises(cz.CzError) as e:
        model.set_match(17)
    assert e.value.code == _lib.CZ_ERR_INVALID
    model.close()


def test_full_size_match_round_trips(gpu_ctx):
    """SmolLM-135M and RWKV-7 0.1B (random init), byte ids: the fixtures and random bytes through compress_many (each container equal to
    compress of that file alone) and decompress_many, and the predictions of one file against the restatement"""
    import corpus

    datas = [corpus.load("alphabet.txt")[:3000], corpus.load("alice29.txt")[:4096], corpus.load("enwik8_3mib")[:4096],
             corpus.high_entropy_stream(2048)]
    for cfg in (cz.SMOLLM_135M, cz.RWKV7_0P1B):
        model = cz.Model(gpu_ctx, cfg).random_init(0, 0.02, 0.02)
        many = codec.compress_many(model, datas, n_segments=16, match_order=4)
        assert many[2] == codec.compress(model, datas[2], n_segments=16, match_order=4)
        assert codec.decompress_many(model, many) == datas
        assert codec.decompress(model, many[1]) == datas[1]
        ids = np.frombuffer(datas[2], np.uint8).astype(np.uint32)
        seg = cz.split_segments(ids.shape[0], 16)
        _check_call(gpu_ctx, model, ids, seg, 4)
        model.close()


def test_full_size_match_compression(gpu_ctx):
    """random-init SmolLM-135M, byte ids, K = 4, one segment (encode only): the alphabet codes under 0.1 bits/byte, 1 MiB of the enwik8
    stand-in to at most 0.6x the match-off container, 1 MiB of random bytes to at most the match-off container + 64 bytes"""
    import corpus

    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    alpha = corpus.load("alphabet.txt")
    blob = codec.compress(model, alpha, match_order=4)
    assert container.read_container(blob)[0]["match_order"] == 4
    assert 8 * len(blob) / len(alpha) < 0.1
    for data, check in ((corpus.load("enwik8_3mib")[: 1 << 20], lambda on, off: on <= 0.6 * off),
                        (corpus.high_entropy_stream(1 << 20), lambda on, off: on <= off + 64)):
        on, off = len(codec.compress(model, data, match_order=4)), len(codec.compress(model, data))
        print(f"match on {on} / off {off} bytes ({on / off:.3f})")
        assert check(on, off), (on, off)
    model.close()
