"""GPU suite for preset dictionaries (cz_model_set_dictionary): a segment coded under dictionary D has, bit for bit, the intervals and
entropies of the last |T| tokens of D ++ T coded without one, on SmolLM (both engines) and RWKV-7 (literal escapes in D and T); payloads
are the coder lanes of those intervals; round trips through compress / decompress and the many-file paths, including the zero-width
fallbacks; digests; a cleared dictionary changes nothing; errors are returned, not crashes."""
import os
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
from candlezip_b200 import _lib, codec, container
from test_gpu_pdf_floor import _PairTokenizer, _peaky

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
DICT_SIZES = [1, 511, 512, 513, 1500]


def _rwkv_tiny(gpu_ctx):
    from rwkv7_weights import RWKV7_TINY, make_weights

    m = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        m.set_tensor(name, arr)
    return m


def _check_equivalence(gpu_ctx, model, ids, dic, n_segments, **kw):
    """analyze(T, dictionary=D) against analyze(D ++ T_g)[|D|:] for every segment g, and each payload against the coder lanes of its
    intervals"""
    r = model.analyze(ids, n_segments=n_segments, dictionary=dic, **kw)
    seg = r["seg_start"]
    nd = len(dic)
    for g in range(len(seg) - 1):
        a, b = int(seg[g]), int(seg[g + 1])
        ref = model.analyze(np.concatenate([dic, ids[a:b]]).astype(np.uint32), **kw)
        for k in ("c_lo", "c_hi"):
            assert np.array_equal(r[k][a:b], ref[k][nd:]), (k, g, nd, np.nonzero(r[k][a:b] != ref[k][nd:])[0][:5])
        assert np.array_equal(r["entropy"][a:b].view(np.uint64), ref["entropy"][nd:].view(np.uint64)), (g, nd)
        assert int(r["first_zw"][g]) == _lib.NO_ZERO_WIDTH
        lanes = gpu_ctx.ac_encode_lanes(r["c_lo"][a:b], r["c_hi"][a:b], np.array([0, b - a], np.uint64))
        assert r["payloads"][g] == lanes[0], (g, nd)
    return r


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_TCGEN05, _lib.CZ_ENGINE_SIMT])
def test_dictionary_equivalence_smollm_tiny(gpu_ctx, engine):
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(5, 0.05, 0.05)
    rng = np.random.default_rng(engine)
    ids = rng.integers(0, cz.SMOLLM_TINY["vocab"], 1400).astype(np.uint32)
    for nd in DICT_SIZES:
        dic = rng.integers(0, cz.SMOLLM_TINY["vocab"], nd).astype(np.uint32)
        for reprime in (512, 7):
            _check_equivalence(gpu_ctx, model, ids, dic, 3, reprime_interval=reprime)
    # one segment, a small context: the prime of the chunk in which D ends is cut to the context window
    _check_equivalence(gpu_ctx, model, ids[:700], rng.integers(0, 1024, 600).astype(np.uint32), 1, context=100, reprime_interval=64)
    model.close()


def test_dictionary_equivalence_rwkv7_tiny(gpu_ctx):
    """literal escapes in T and in D, a D of literal escapes only, and slabs smaller than D (the dictionary then runs in several)"""
    model = _rwkv_tiny(gpu_ctx)
    V = model.cfg["vocab"]
    rng = np.random.default_rng(3)
    ids = rng.integers(0, V + 256, 1200).astype(np.uint32)
    for nd in DICT_SIZES:
        dic = rng.integers(0, V + 256, nd).astype(np.uint32)
        _check_equivalence(gpu_ctx, model, ids, dic, 3)
    lit = (V + rng.integers(0, 256, 40)).astype(np.uint32)
    _check_equivalence(gpu_ctx, model, ids, lit, 3)
    _check_equivalence(gpu_ctx, model, ids, np.concatenate([lit, [5], lit]).astype(np.uint32), 2)
    _check_equivalence(gpu_ctx, model, ids, rng.integers(0, V, 1500).astype(np.uint32), 4, max_batch_tokens=256)
    model.close()


def _text_files(seed, n_files=12):
    import corpus

    rng = np.random.default_rng(seed)
    text = corpus.load("alice29.txt")
    out = []
    for k in range(n_files):
        n = [0, 1, 40, 300, 700, 1500][k % 6]
        a = int(rng.integers(0, len(text) - n))
        out.append(text[a : a + n])
    return out


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_TCGEN05, _lib.CZ_ENGINE_SIMT])
def test_dictionary_round_trips_and_batches_tiny(gpu_ctx, engine):
    import corpus

    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(5, 0.05, 0.05)
    dic = corpus.load("asyoulik.txt")[:700]
    datas = _text_files(engine)
    for nseg in (1, 3):
        many = codec.compress_many(model, datas, n_segments=nseg, dictionary=dic)
        for i, d in enumerate(datas):
            one = codec.compress(model, d, n_segments=nseg, dictionary=dic)
            assert many[i] == one, (nseg, i)
            if d:
                assert container.read_container(one)[0]["reserved_flags"] & _lib.CZ_FLAG_DICTIONARY
                assert codec.decompress(model, one, dictionary=dic) == d
        assert codec.decompress_many(model, many, dictionary=dic) == datas
        assert codec.decompress_many(model, many, max_streams=3, dictionary=dic) == datas
    model.close()


def test_dictionary_round_trips_rwkv7_tiny(gpu_ctx):
    model = _rwkv_tiny(gpu_ctx)
    vocab = {bytes([c]): i + 1 for i, c in enumerate(b"abcdefghijklmnopqrstuvwxyz .,")}
    vocab.update({w: 200 + k for k, w in enumerate([b"th", b"he", b"in", b"er", b"an", b"the", b"ing"])})
    tok = codec.RwkvTokenizer(vocab)
    datas = [d.lower() for d in _text_files(9)]  # capitals, digits and punctuation outside the vocabulary go out as literal escapes
    for dic in (b"the thing, The Other Thing", b"ABC!?", b"q"):
        for nseg in (1, 3):
            many = codec.compress_many(model, datas, tok, n_segments=nseg, dictionary=dic)
            assert many == [codec.compress(model, d, tok, n_segments=nseg, dictionary=dic) for d in datas], (dic, nseg)
            assert codec.decompress_many(model, many, tok, dictionary=dic) == datas
            assert codec.decompress_many(model, many, tok, max_streams=3, dictionary=dic) == datas
            assert codec.decompress(model, many[4], tok, dictionary=dic) == datas[4]
    model.close()


@pytest.mark.parametrize("policy", ["stored", "floor"])
def test_dictionary_zero_width_fallbacks(gpu_ctx, policy):
    """the peaky model: random tokens are zero-width without the floor, whatever precedes them.  Files fall back by the policy, the
    floored re-code uses the same dictionary, and every container round-trips"""
    model = _peaky(gpu_ctx)
    tok = _PairTokenizer()
    rng = np.random.default_rng(11)
    datas = [tok.decode_bytes(rng.integers(0, 1024, n)) for n in (300, 0, 900, 40)]
    dic = tok.decode_bytes(rng.integers(0, 1024, 520))
    want = _lib.CZ_FLAG_STORED if policy == "stored" else _lib.CZ_FLAG_PDF_FLOOR | _lib.CZ_FLAG_DICTIONARY
    for nseg in (1, 2):
        many = codec.compress_many(model, datas, tok, n_segments=nseg, on_zero_width=policy, dictionary=dic)
        for i, d in enumerate(datas):
            assert many[i] == codec.compress(model, d, tok, n_segments=nseg, on_zero_width=policy, dictionary=dic), (policy, nseg, i)
            flags = container.read_container(many[i])[0]["reserved_flags"] & ~_lib.CZ_FLAG_SEGMENTS
            assert flags == (want if d else _lib.CZ_FLAG_DICTIONARY), (policy, nseg, i, flags)
        assert codec.decompress_many(model, many, tok, dictionary=dic) == datas
        assert codec.decompress_many(model, many, tok, max_streams=3, dictionary=dic) == datas
    model.close()


def test_dictionary_digests_and_cleared_dictionary(gpu_ctx):
    """encode digests equal decode digests under a dictionary (SmolLM, several streams; RWKV-7); a dictionary set and cleared again
    launches and writes exactly what a model that never had one does"""
    rng = np.random.default_rng(2)
    for model in (cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05), _rwkv_tiny(gpu_ctx)):
        V = model.cfg["vocab"]
        lim = V + (256 if model.cfg["arch"] == 1 else 0)
        ids = rng.integers(0, lim, 1100).astype(np.uint32)
        dic = rng.integers(0, lim, 600).astype(np.uint32)
        model.watch_digests(len(ids))
        pays, seg = model.encode(ids, n_segments=3, dictionary=dic)
        enc = model._digests.copy()
        model.watch_digests(len(ids))
        assert np.array_equal(model.decode(pays, seg, dictionary=dic), ids)
        assert np.array_equal(model._digests, enc) and np.any(enc != 0)
        model.watch_digests(0)
        # the same call on a fresh model and on one whose dictionary was cleared
        fresh = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05) if model.cfg["arch"] == 0 else _rwkv_tiny(gpu_ctx)
        fresh.encode(ids[:10])  # (a model's first call prepares its weights)
        counts = []
        for m in (fresh, model):
            if m is model:
                m.set_dictionary(dic)
                m.set_dictionary(None)
            l0 = gpu_ctx.launch_count()
            p, s = m.encode(ids, n_segments=3)
            out = m.decode(p, s)
            counts.append((gpu_ctx.launch_count() - l0, p))
            assert np.array_equal(out, ids)
        assert counts[0] == counts[1]
        assert counts[0][1] != pays  # (the dictionary did change the payloads)
        fresh.close()
        model.close()


def test_dictionary_errors_are_returned(gpu_ctx):
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=_lib.CZ_ENGINE_SIMT).random_init(5, 0.05, 0.05)
    ids = np.arange(50, dtype=np.uint32)
    with pytest.raises(cz.CzError) as e:
        model.encode(ids, dictionary=np.array([1, 2, 5000], np.uint32))
    assert e.value.code == _lib.CZ_ERR_SYMBOL_RANGE and "at index 2" in str(e.value)
    ev = [(10, np.array([7, 8], np.uint32), 0)]
    with pytest.raises(cz.CzError) as e:
        model.encode(ids, events=ev, dictionary=np.array([1, 2], np.uint32))
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    pays, seg = model.encode(ids, events=ev)
    with pytest.raises(cz.CzError) as e:
        model.decode(pays, seg, events=ev, dictionary=np.array([1, 2], np.uint32))
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    # without reprimes the chunk in which a long dictionary ends holds all of it: beyond the attention kernel's sequence length
    long = np.arange(2500, dtype=np.uint32) % 1024
    with pytest.raises(cz.CzError) as e:
        model.encode(ids, reprime_interval=1 << 20, dictionary=long)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    with pytest.raises(cz.CzError) as e:
        model.decode(pays, seg, reprime_interval=1 << 20, dictionary=long)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    # the model still works, without a dictionary (every call above cleared it again)
    assert np.array_equal(model.decode(*model.encode(ids)), ids)
    model.close()


def test_full_size_dictionary(gpu_ctx):
    """SmolLM-135M and RWKV-7 0.1B (random init): equivalence at |D| = 513 over three segments, and a many-file round trip"""
    import corpus

    text = corpus.load("alice29.txt")
    dic_bytes = text[:4096]
    datas = [text[5000 + 700 * k : 5000 + 700 * k + n] for k, n in enumerate([0, 100, 600, 1300, 2500])]
    rng = np.random.default_rng(0)
    for cfg in (cz.SMOLLM_135M, cz.RWKV7_0P1B):
        model = cz.Model(gpu_ctx, cfg).random_init(0, 0.02, 0.02)
        ids = rng.integers(0, cfg["vocab"], 1600).astype(np.uint32)
        _check_equivalence(gpu_ctx, model, ids, rng.integers(0, cfg["vocab"], 513).astype(np.uint32), 3)
        many = codec.compress_many(model, datas, n_segments=2, dictionary=dic_bytes)
        assert many[3] == codec.compress(model, datas[3], n_segments=2, dictionary=dic_bytes)
        assert codec.decompress_many(model, many, dictionary=dic_bytes) == datas
        model.close()
