"""GPU suite for the many-file codec (codec.compress_many / decompress_many) and the per-segment zero-width report
(cz_model_set_zero_width_out): every container equal byte for byte to coding the file alone, round trips through lock-step waves of
any size, the report against what cz_encode names for a segment coded alone, RWKV-7, mixed containers, and the CLI."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
from candlezip_b200 import _lib, codec, container
from test_gpu_pdf_floor import _greedy_with_one_surprise, _PairTokenizer, _peaky

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
NONE = _lib.NO_ZERO_WIDTH
LENGTHS = [0, 1, 2, 511, 512, 513, 1023, 1500, 3000]


def _files(seed):
    """about 40 files of LENGTHS bytes: random bytes and corpus slices"""
    import corpus

    rng = np.random.default_rng(seed)
    text = corpus.load("alice29.txt") + corpus.load("asyoulik.txt")
    out = []
    for k in range(40):
        n = LENGTHS[k % len(LENGTHS)]
        if k % 2:
            out.append(bytes(rng.integers(0, 256, n, dtype=np.uint8)))
        else:
            a = int(rng.integers(0, len(text) - n))
            out.append(text[a : a + n])
    return out


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_TCGEN05, _lib.CZ_ENGINE_SIMT])
def test_tiny_smollm_batch_equals_singles_and_round_trips(gpu_ctx, engine):
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(5, 0.05, 0.05)
    datas = _files(engine)
    for nseg in (1, 3):
        many = codec.compress_many(model, datas, n_segments=nseg)
        assert len(many) == len(datas)
        for i, d in enumerate(datas):
            assert many[i] == codec.compress(model, d, n_segments=nseg), (nseg, i, len(d))
        assert codec.decompress_many(model, many) == datas, nseg
        assert codec.decompress_many(model, many, max_streams=3) == datas, nseg
    model.close()


def _first_zw_alone(model, ids):
    """the index cz_encode names when `ids` is coded alone as one segment, or NONE"""
    try:
        model.encode(ids)
        return NONE
    except cz.CzError as e:
        assert e.code == _lib.CZ_ERR_ZERO_WIDTH
        return int(re.search(r"at coded index (\d+)", str(e)).group(1))


def test_peaky_sink_and_fallbacks(gpu_ctx):
    """the peaky tiny model: files with one surprise token (zero-width unfloored) mixed with clean ones.  The sink's per-segment index
    is the index cz_encode names for that segment alone and the clean segments' payloads are their payloads alone; without the sink the
    batched call still fails; under both policies every container equals compress() alone and decompresses"""
    model = _peaky(gpu_ctx)
    tok = _PairTokenizer()
    specs = [(300, -1), (1200, 700), (600, -1), (900, 5), (1500, 1400), (40, -1), (0, -1), (513, 512)]
    id_lists = [_greedy_with_one_surprise(model, n, at) for n, at in specs]
    datas = [tok.decode_bytes(x) for x in id_lists]
    for nseg in (1, 3):
        seg, ranges, _ = codec.pack_segments([len(x) for x in id_lists], nseg)
        ids = np.concatenate(id_lists).astype(np.uint32)
        with pytest.raises(cz.CzError) as e:
            model.encode(ids, seg_start=seg)
        assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH
        pays, _, zw = model.encode(ids, seg_start=seg, zero_width_out=True)
        assert zw.shape[0] == len(seg) - 1
        for g in range(len(seg) - 1):
            part = ids[int(seg[g]) : int(seg[g + 1])]
            assert int(zw[g]) == _first_zw_alone(model, part), (nseg, g)
            if zw[g] == NONE:
                assert model.encode(part)[0] == [pays[g]], (nseg, g)
        bad = codec.zero_width_files(ranges, zw)
        surprised = [i for i, (n, at) in enumerate(specs) if 0 <= at < n]
        # (a later segment restarts from BOS, where a greedy token of the whole file may be zero-width too)
        assert bad == surprised if nseg == 1 else set(surprised) <= set(bad), (nseg, bad)
        for policy in ("stored", "floor"):
            many = codec.compress_many(model, datas, tok, n_segments=nseg, on_zero_width=policy)
            for i, d in enumerate(datas):
                assert many[i] == codec.compress(model, d, tok, n_segments=nseg, on_zero_width=policy), (nseg, policy, i)
            want = _lib.CZ_FLAG_STORED if policy == "stored" else _lib.CZ_FLAG_PDF_FLOOR
            flags = [container.read_container(b)[0]["reserved_flags"] & (_lib.CZ_FLAG_STORED | _lib.CZ_FLAG_PDF_FLOOR) for b in many]
            assert flags == [want if i in bad else 0 for i in range(len(datas))], (nseg, policy, flags)
            assert codec.decompress_many(model, many, tok) == datas, (nseg, policy)
    # the C entry point's argument checks
    buf = np.zeros(2, np.uint64)
    assert _lib.lib.cz_model_set_zero_width_out(model._h, buf.ctypes.data_as(_lib.u64p), 0) == _lib.CZ_ERR_INVALID
    _lib.check(_lib.lib.cz_model_set_zero_width_out(model._h, buf.ctypes.data_as(_lib.u64p), 2))
    with pytest.raises(cz.CzError) as e:
        model.encode(np.arange(30, dtype=np.uint32), n_segments=3)
    assert e.value.code == _lib.CZ_ERR_INVALID
    _lib.check(_lib.lib.cz_model_set_zero_width_out(model._h, None, 0))
    with pytest.raises(cz.CzError) as e:
        model.encode(id_lists[1])
    assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH
    model.close()


def _rwkv(gpu_ctx):
    from rwkv7_weights import RWKV7_TINY, make_weights

    m = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        m.set_tensor(name, arr)
    return m


def test_rwkv7_batch_equals_singles(gpu_ctx):
    """RWKV-7 tiny with an RwkvTokenizer (files it cannot express go out as literal escapes): batch == singles, round trips through
    waves, and the sink reports no zero-width segment"""
    model = _rwkv(gpu_ctx)
    vocab = {bytes([c]): i + 1 for i, c in enumerate(b"abcdefghijklmnopqrstuvwxyz .,")}
    vocab.update({w: 200 + k for k, w in enumerate([b"th", b"he", b"in", b"er", b"an", b"the", b"ing"])})
    tok = codec.RwkvTokenizer(vocab)
    rng = np.random.default_rng(4)
    words = [b"the", b"thing", b"in", b"an", b"other", b"rain", b"bring", b"he"]
    datas = []
    for k in range(12):
        n = [0, 1, 30, 200, 700][k % 5]
        text = b" ".join(words[int(j)] for j in rng.integers(0, len(words), n))[:n]
        datas.append(text if k % 3 else text + b"\x00\xff7" + bytes(rng.integers(0, 256, n // 4, dtype=np.uint8)))
    for nseg in (1, 3):
        many = codec.compress_many(model, datas, tok, n_segments=nseg)
        for i, d in enumerate(datas):
            assert many[i] == codec.compress(model, d, tok, n_segments=nseg), (nseg, i)
        assert codec.decompress_many(model, many, tok) == datas
        assert codec.decompress_many(model, many, tok, max_streams=2) == datas
    ids = [codec.tokenize(model, d, tok) for d in datas]
    seg, _, _ = codec.pack_segments([len(x) for x in ids], 3)
    _, _, zw = model.encode(np.concatenate(ids).astype(np.uint32), seg_start=seg, zero_width_out=True)
    assert zw.shape[0] == len(seg) - 1 and np.all(zw == NONE)
    model.close()


def test_decompress_many_mixed_containers(gpu_ctx):
    """v2 single-stream, SEG1, STORED, PDF_FLOOR and two (context, reprime) settings in one call; a gated and a corrupted container
    each raise naming their index"""
    import corpus

    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
    text = corpus.load("asyoulik.txt")
    datas = [text[a : a + n] for a, n in ((0, 700), (900, 250), (4000, 1100), (7000, 800))]
    blobs, want = [], []
    for ctx_, rp in ((512, 512), (256, 256)):
        for nseg in (1, 2):
            for d in datas[:3]:
                blobs.append(codec.compress(model, d, n_segments=nseg, context=ctx_, reprime_interval=rp))
                want.append(d)
        d = datas[3]
        fields = codec.header_fields(model, d, len(d), 0, ctx_, rp, b"\0" * 16, b"\0" * 16)
        blobs.append(codec.stored_container(fields, b"model.safetensors", d))
        pays, seg = model.encode(codec.tokenize(model, d, codec.ByteTokenizer()), n_segments=2, context=ctx_, reprime_interval=rp,
                                 pdf_floor=True)
        blobs.append(codec.coded_container(model, dict(fields, reserved_flags=_lib.CZ_FLAG_PDF_FLOOR), b"model.safetensors", pays, seg))
        want += [d, d]
    blobs.append(codec.compress(model, b""))
    want.append(b"")
    flags = [container.read_container(b)[0]["reserved_flags"] for b in blobs]
    assert sum(1 for f in flags if f & _lib.CZ_FLAG_SEGMENTS and not f & (_lib.CZ_FLAG_STORED | _lib.CZ_FLAG_PDF_FLOOR)) == 6
    assert sum(1 for f in flags if f == 0) == 7  # v2 single stream (+ the empty file)
    assert codec.decompress_many(model, blobs) == want
    assert codec.decompress_many(model, blobs, max_streams=4) == want
    assert [codec.decompress(model, b) for b in blobs] == want
    f, rep, _, _, _, pays = container.read_container(blobs[0])
    gated = container.write_container(dict(f), rep, pays, gates=[0, 1])
    with pytest.raises(ValueError, match=r"^blob 3: gated"):
        codec.decompress_many(model, blobs[:3] + [gated])
    corrupt = bytearray(blobs[1])
    corrupt[-5] ^= 0x40
    with pytest.raises(ValueError, match=r"^blob 2: decoded bytes do not match"):
        codec.decompress_many(model, [blobs[0], blobs[2], bytes(corrupt)])
    model.close()


def test_full_size_smollm_batch(gpu_ctx):
    """SmolLM-135M shape: 16 files of about 1,300 tokens, batch == singles, round trip"""
    import corpus

    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    text = corpus.load("alice29.txt")
    rng = np.random.default_rng(8)
    datas = [text[int(a) : int(a) + 1250 + 7 * k] for k, a in enumerate(rng.integers(0, len(text) - 1400, 16))]
    many = codec.compress_many(model, datas)
    for i, d in enumerate(datas):
        assert many[i] == codec.compress(model, d), i
    assert codec.decompress_many(model, many) == datas
    model.close()


def test_cli_many(gpu_ctx, tmp_path):
    """compress-many / decompress-many on three files: each .canz is what compress writes for that file, and they round-trip"""
    import corpus

    text = corpus.load("alice29.txt")
    names = ["a.txt", "b.bin", "c.txt"]
    datas = [text[:900], bytes(np.random.default_rng(1).integers(0, 256, 300, dtype=np.uint8)), text[5000:5001]]
    for nm, d in zip(names, datas):
        (tmp_path / nm).write_bytes(d)
    out = tmp_path / "out"
    r = subprocess.run([sys.executable, "-m", "candlezip_b200", "compress-many", *[str(tmp_path / nm) for nm in names], "--out-dir", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-800:]
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    for nm, d in zip(names, datas):
        assert (out / (nm + ".canz")).read_bytes() == codec.compress(model, d), nm
    model.close()
    back = tmp_path / "back"
    r = subprocess.run([sys.executable, "-m", "candlezip_b200", "decompress-many", *[str(out / (nm + ".canz")) for nm in names], "--out-dir",
                        str(back), "--max-streams", "2"], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-800:]
    for nm, d in zip(names, datas):
        assert (back / (nm + ".canz.out")).read_bytes() == d, nm
