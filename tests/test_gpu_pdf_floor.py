"""GPU suite for the floored SmolLM coding alphabet (CZ_CDF_SMOLLM_FLOOR, cz_model_set_pdf_floor, CZ_FLAG_PDF_FLOOR): the K1 kernels
bit-exact against the oracle's quantize_pdf_to_cdf(softmax_pdf_floor(.)), the coding loop on a model that meets zero-width symbols
without the floor, invariance of the mode-2 bytes, and the file-level / CLI surface."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
from candlezip_b200 import _lib
from test_cpu_pdf_floor import adversarial_logits, cdf_floor

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
FLOOR = _lib.CZ_CDF_SMOLLM_FLOOR


def _peaky(gpu_ctx, engine=_lib.CZ_ENGINE_TCGEN05, cfg=cz.SMOLLM_TINY):
    return cz.Model(gpu_ctx, cfg, engine=engine).random_init(5, 0.05, 1.5)  # logits std ~ 20: random tokens are zero-width unfloored


def _check_k1(gpu_ctx, logits, syms, rng):
    """cz_cdf_bounds / cz_cdf_search / cz_xe_bits_cols in mode 2 against the oracle, column by column"""
    v, m = logits.shape
    lo, hi = gpu_ctx.cdf_bounds(logits, syms, FLOOR)
    assert np.all(hi > lo), "a coded symbol got an empty interval"
    cdfs = [cdf_floor(logits[:, j]) for j in range(m)]
    want_lo = np.array([c[s] for c, s in zip(cdfs, syms)], np.uint32)
    want_hi = np.array([c[s + 1] for c, s in zip(cdfs, syms)], np.uint32)
    bad = np.nonzero((lo != want_lo) | (hi != want_hi))[0]
    assert bad.size == 0, (v, m, bad[:5], syms[bad[:5]])
    # search: the lower bound of a symbol's interval, a random value inside it, and values anywhere
    for values in (want_lo, (want_lo + (rng.random(m) * (want_hi - want_lo)).astype(np.uint32)).astype(np.uint32),
                   rng.integers(0, 1 << 30, m).astype(np.uint32)):
        s, slo, shi = gpu_ctx.cdf_search(logits, values, FLOOR)
        ws = np.array([np.searchsorted(c, x, side="right") - 1 for c, x in zip(cdfs, values)], np.uint32)
        assert np.array_equal(s, ws), (v, m)
        assert np.array_equal(slo, [c[k] for c, k in zip(cdfs, ws)]) and np.array_equal(shi, [c[k + 1] for c, k in zip(cdfs, ws)])
    # XE: mode 2 is mode 0 there (cz_xe_bits_cols already floors SmolLM), bit for bit
    xe2 = gpu_ctx.xe_bits_cols(logits, syms, FLOOR)
    assert np.array_equal(xe2.view(np.uint64), gpu_ctx.xe_bits_cols(logits, syms, 0).view(np.uint64))
    for j in range(min(m, 40)):
        want = -np.log2(max(oracle.softmax_pdf_floor(logits[:, j])[syms[j]], 1e-300))
        assert abs(xe2[j] - want) <= 1e-12 * max(1.0, abs(want)), j


@pytest.mark.parametrize("v", [1024, 4099, 49152])
def test_k1_floor_mode_bit_exact_tma_direct_and_vector_widths(gpu_ctx, v):
    """every kernel family of mode 2: the TMA-staged stats pass (>= 256 aligned columns), the direct-load stats kernel (40 columns, and
    CZ_CDF_NCOL = 1 / 2 / 4), the warp-per-column prefix walk, the warp search; a column whose entries are mostly > 87 below the max
    (the fast expf's conversion fallback); symbols at both ends of the alphabet; cz_cdf_full"""
    rng = np.random.default_rng(v)
    try:
        for ncol in (0, 1, 2, 4):
            if ncol:
                os.environ["CZ_CDF_NCOL"] = str(ncol)
            for m in ((40, 260, 1024) if v < 49152 or ncol in (0, 2) else (260,)):
                logits = adversarial_logits(rng, v, m)
                logits[:, m // 2] = rng.normal(0, 30, v)
                syms = rng.integers(0, v, m).astype(np.uint32)
                syms[:6] = [0, v - 1, 1, v - 2, 5, v // 3]
                _check_k1(gpu_ctx, logits, syms, rng)
            os.environ.pop("CZ_CDF_NCOL", None)
    finally:
        os.environ.pop("CZ_CDF_NCOL", None)
    if v == 1024:  # more columns than the warp search takes: the thread-per-column search (cdf_cols_kernel)
        logits = adversarial_logits(rng, v, 8200)
        values = rng.integers(0, 1 << 30, 8200).astype(np.uint32)
        s, slo, shi = gpu_ctx.cdf_search(logits, values, FLOOR)
        for j in range(8200):
            c = cdf_floor(logits[:, j])
            k = np.searchsorted(c, values[j], side="right") - 1
            assert (s[j], slo[j], shi[j]) == (k, c[k], c[k + 1]), j
    logits = adversarial_logits(rng, v, 8)
    for j in (1, 3, 5, 7):
        assert np.array_equal(gpu_ctx.cdf_full(logits[:, j], FLOOR), cdf_floor(logits[:, j])), j
    with pytest.raises(cz.CzError) as e:
        gpu_ctx.cdf_bounds(logits, np.zeros(8, np.uint32), 3)
    assert e.value.code == _lib.CZ_ERR_INVALID
    with pytest.raises(cz.CzError) as e:
        gpu_ctx.cdf_full(logits[:, 0], 3)
    assert e.value.code == _lib.CZ_ERR_INVALID


def test_floor_prefix_walk_through_the_ecache_and_its_fallback(gpu_ctx):
    """mode 2's prefix walk (a) through the e-cache, (b) when the batch does not fit it, (c) with the cache disabled: same bounds as the
    oracle every time, and the state hook says which of the three ran"""

    def state():
        st, g = C.c_int(), C.c_uint64()
        _lib.check(_lib.lib.cz_test_cdf_ecache_state(gpu_ctx._h, C.byref(st), C.byref(g)))
        return st.value

    rng = np.random.default_rng(31)
    v = 4099
    try:
        for m in (260, 1024):
            logits = adversarial_logits(rng, v, m)
            logits[:, m // 3] = rng.normal(0, 30, v)
            heavy = np.minimum((rng.random(m) ** 6 * v).astype(np.uint32), v - 1)
            heavy[:4] = [0, 1, 8, v - 1]
            uniform = rng.integers(0, v, m).astype(np.uint32)
            cdfs = [cdf_floor(logits[:, j]) for j in range(m)]
            for name, frac, expect in [("heavy", None, 1), ("uniform", None, 0), ("uniform", "1.0", 1), ("heavy", "off", -1)]:
                os.environ.pop("CZ_CDF_ECACHE_FRAC", None)
                os.environ.pop("CZ_CDF_NO_ECACHE", None)
                if frac == "off":
                    os.environ["CZ_CDF_NO_ECACHE"] = "1"
                elif frac:
                    os.environ["CZ_CDF_ECACHE_FRAC"] = frac
                syms = heavy if name == "heavy" else uniform
                lo, hi = gpu_ctx.cdf_bounds(logits, syms, FLOOR)
                assert state() == expect, (m, name, frac)
                assert np.array_equal(lo, [c[s] for c, s in zip(cdfs, syms)]) and np.array_equal(hi, [c[s + 1] for c, s in zip(cdfs, syms)]), (m, name)
                assert np.all(hi > lo)
    finally:
        os.environ.pop("CZ_CDF_ECACHE_FRAC", None)
        os.environ.pop("CZ_CDF_NO_ECACHE", None)


def _oracle_payload(model, ids, n0):
    """the oracle coder over oracle mode-2 bounds of segment 0 (ids[:n0]), from the GPU's teacher-forced logits, chunk by chunk
    (every reprime of the schedule, cz_schedule_chunks)"""
    cap = 64
    first, ncod, pst, plen = (np.zeros(cap, np.uint64), np.zeros(cap, np.uint32), np.zeros(cap, np.uint64), np.zeros(cap, np.uint32))
    k = _lib.lib.cz_schedule_chunks(n0, 512, 512, first.ctypes.data_as(_lib.u64p), ncod.ctypes.data_as(_lib.u32p), pst.ctypes.data_as(_lib.u64p),
                                    plen.ctypes.data_as(_lib.u32p), cap)
    seq = np.concatenate([[0], ids[:n0]]).astype(np.uint32)
    bounds = []
    for c in range(k):
        f, n, p0, pl = int(first[c]), int(ncod[c]), int(pst[c]), int(plen[c])
        lg = model.chunk_logits(seq[p0:p0 + pl], ids[f:f + n])
        for j in range(n):
            cdf = cdf_floor(lg[j])
            bounds.append((int(cdf[ids[f + j]]), int(cdf[ids[f + j] + 1])))
    assert len(bounds) == n0 and all(h > l for l, h in bounds)
    return oracle.ac_encode(bounds)


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_TCGEN05, _lib.CZ_ENGINE_SIMT])
def test_peaky_model_codes_with_the_floor(gpu_ctx, engine):
    """the peaky tiny model (random tokens are zero-width unfloored): mode 0 refuses, mode 2 encodes, segment 0's bytes are the oracle
    coder's over oracle mode-2 bounds (across reprimes), and the lock-step decoder gets the tokens back"""
    model = _peaky(gpu_ctx, engine)
    rng = np.random.default_rng(engine)
    for n in (700, 1700, 2300):
        ids = rng.integers(0, 1024, n).astype(np.uint32)
        for nseg in (1, 3, 5):
            with pytest.raises(cz.CzError) as e:
                model.encode(ids, n_segments=nseg)
            assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH
            pays, seg = model.encode(ids, n_segments=nseg, pdf_floor=True)
            if nseg != 3:  # (segment 0 of 1 and 5 segments: 700 .. 2300 and 140 .. 460 tokens)
                assert pays[0] == _oracle_payload(model, ids, int(seg[1])), (n, nseg)
            assert np.array_equal(model.decode(pays, seg, pdf_floor=True), ids), (n, nseg)


def test_floor_mode_bytes_are_invariant(gpu_ctx):
    """mode 2's bytes do not depend on the wave size or on the other segments; on a model without zero-width tokens the flag changes
    neither the logits (digests, encode == decode) nor cz_xe_bits, and costs at most log2(1 + V 2^-29) bits per token"""
    model = _peaky(gpu_ctx)
    rng = np.random.default_rng(17)
    ids = rng.integers(0, 1024, 2100).astype(np.uint32)
    pays, seg = model.encode(ids, n_segments=3, pdf_floor=True)
    for mbt in (700, 1500):
        assert model.encode(ids, n_segments=3, pdf_floor=True, max_batch_tokens=mbt)[0] == pays, mbt
    for g in range(3):
        a, b = int(seg[g]), int(seg[g + 1])
        assert model.encode(ids[a:b], pdf_floor=True)[0] == [pays[g]], g
    model.close()

    import corpus

    flat = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
    ids = np.frombuffer(corpus.load("alice29.txt")[:1700], np.uint8).astype(np.uint32)
    dig = flat.watch_digests(len(ids))
    p0, s0 = flat.encode(ids, n_segments=3)
    d0 = dig.copy()
    dig[:] = 0
    p2, s2 = flat.encode(ids, n_segments=3, pdf_floor=True)
    assert np.array_equal(dig, d0), "the floor changed the logits"
    dig[:] = 0
    assert np.array_equal(flat.decode(p2, s2, pdf_floor=True), ids) and np.array_equal(dig, d0), "decode digests differ"
    flat.watch_digests(0)
    n0, n2 = sum(map(len, p0)), sum(map(len, p2))
    assert n2 <= n0 * 1.0001 + 2, (n0, n2)
    jobs = [(ids[:300], ids[300:420]), (ids[7:511], ids[511:600])]
    xe0 = flat.xe_bits(jobs)
    flat.set_pdf_floor(True)
    assert np.array_equal(flat.xe_bits(jobs).view(np.uint64), xe0.view(np.uint64))
    flat.set_pdf_floor(False)


def test_full_size_floor_round_trip(gpu_ctx):
    """SmolLM-135M shape (V = 49,152), peaky random init, 1,300 tokens in 2 segments: mode 2 round-trips and segment 0's bytes (two
    chunks: 512 + a reprimed 138) are the oracle coder's over oracle mode-2 bounds"""
    model = _peaky(gpu_ctx, cfg=cz.SMOLLM_135M)
    ids = np.random.default_rng(23).integers(0, 49152, 1300).astype(np.uint32)
    pays, seg = model.encode(ids, n_segments=2, pdf_floor=True)
    assert np.array_equal(model.decode(pays, seg, pdf_floor=True), ids)
    assert pays[0] == _oracle_payload(model, ids, int(seg[1]))


class _PairTokenizer:
    """two bytes per token (little-endian id): lets a test file hold any of the tiny model's 1,024 ids"""

    def encode_bytes(self, data):
        return np.frombuffer(data, "<u2").astype(np.uint32)

    def decode_bytes(self, ids):
        return np.asarray(ids, "<u2").tobytes()


def _greedy_with_one_surprise(model, n, at):
    """tokens the model predicts (argmax, with the coder's reprime schedule) except token `at`, its least likely one"""
    s = model.session()
    logits = s.step_logits_tensor(0)
    seq = [0]
    for i in range(n):
        if i > 0 and i % 512 == 0 and s.index_pos() >= 511:
            logits = s.reprime_with_history_and_get_last_logits_tensor(np.asarray(seq[-511:], np.uint32))
        t = int(np.argmin(logits) if i == at else np.argmax(logits))
        seq.append(t)
        logits = s.step_logits_tensor(t)
    s.close()
    return np.asarray(seq[1:], np.uint32)


def test_file_level_floor_fallback_and_cli(gpu_ctx, tmp_path):
    """compress(on_zero_width="floor"): a file the unfloored coder cannot code is coded with the floor (PDF_FLOOR, not STORED),
    comes out smaller than the input and decompresses to it; a file without such a token gives the default container byte for byte;
    the CLI's self-test takes --on-zero-width floor; an RWKV-7 model refuses the switch"""
    from candlezip_b200 import codec, container

    model = _peaky(gpu_ctx)
    tok = _PairTokenizer()
    ids = _greedy_with_one_surprise(model, 1200, 700)
    data = tok.decode_bytes(ids)
    with pytest.raises(cz.CzError) as e:
        model.encode(ids)
    assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH
    for nseg in (1, 3):
        blob = codec.compress(model, data, tok, nseg, on_zero_width="floor")
        flags = container.read_container(blob)[0]["reserved_flags"]
        assert flags & _lib.CZ_FLAG_PDF_FLOOR and not flags & _lib.CZ_FLAG_STORED and len(blob) < len(data), (nseg, len(blob))
        assert codec.decompress(model, blob, tok) == data
        stored = codec.compress(model, data, tok, nseg)
        assert container.read_container(stored)[0]["reserved_flags"] & _lib.CZ_FLAG_STORED and codec.decompress(model, stored, tok) == data
    model.close()
    flat = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
    plain = bytes(np.random.default_rng(1).integers(0, 256, 3000, dtype=np.uint8))
    for nseg in (1, 4):
        a = codec.compress(flat, plain, n_segments=nseg)
        assert codec.compress(flat, plain, n_segments=nseg, on_zero_width="floor") == a
        assert container.read_container(a)[0]["reserved_flags"] & (_lib.CZ_FLAG_STORED | _lib.CZ_FLAG_PDF_FLOOR) == 0
    src = tmp_path / "alice_head.txt"
    import corpus

    src.write_bytes(corpus.load("alice29.txt")[:1500])
    r = subprocess.run([sys.executable, "-m", "candlezip_b200", "self-test", str(src), "--on-zero-width", "floor", "--segments", "2"], cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "roundtrip OK" in r.stdout, (r.stdout, r.stderr[-800:])
    from rwkv7_weights import RWKV7_TINY, make_weights

    rm = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        rm.set_tensor(name, arr)
    rid = np.random.default_rng(2).integers(0, RWKV7_TINY["vocab"], 50).astype(np.uint32)
    with pytest.raises(cz.CzError) as e:
        rm.encode(rid, pdf_floor=True)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED
    assert _lib.lib.cz_model_set_pdf_floor(rm._h, 1) == _lib.CZ_ERR_UNSUPPORTED
    rm.encode(rid)
