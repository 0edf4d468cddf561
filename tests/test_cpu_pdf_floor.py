"""CPU suite for the floored SmolLM coding alphabet (CZ_CDF_SMOLLM_FLOOR = quantize_pdf_to_cdf(softmax_pdf_floor(logits, 2^-29)),
src/main.rs:758-767 + 803-824): its reference CDF, the reference coding loop with it, and the container flag CZ_FLAG_PDF_FLOOR.

The reference CDF is composed from the oracle's own softmax_pdf_floor and quantize_pdf_to_cdf (the functions the RWKV alphabet and
the gate XE are checked with); the GPU suite (test_gpu_pdf_floor.py) imports cdf_floor / encode_loop / decode_loop from here."""
import os

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P_FLOOR = 2.0 ** -29
TOTAL = 1 << 30


def cdf_floor(logits):
    """CZ_CDF_SMOLLM_FLOOR's CDF of one logits vector (V + 1 entries), through the oracle"""
    pdf = oracle.softmax_pdf_floor(logits)
    cdf = np.empty(pdf.shape[0] + 1, np.uint32)
    oracle.lib.czo_quantize_pdf_to_cdf(pdf.ctypes.data_as(oracle.f64p), pdf.shape[0], cdf.ctypes.data_as(oracle.u32p))
    return cdf


def cdf_floor_numpy(logits):
    """the same CDF restated in numpy: sequential f64 sums (np.cumsum adds left to right), glibc's expf through the oracle"""
    x = np.asarray(logits, np.float32)
    mx = np.float32(-np.inf)
    for v in x:  # NaN-ignoring `if v > max`
        if v > mx:
            mx = v
    d = (x - mx).astype(np.float32)
    e = np.array([oracle.lib.czo_expf(float(a)) for a in d], np.float64)
    S = np.cumsum(e)[-1]
    p = np.maximum(e / S, P_FLOOR)
    q = p / np.cumsum(p)[-1]
    acc = np.cumsum(q)
    c = np.clip(np.floor(acc * TOTAL), 0, TOTAL)
    c = np.maximum.accumulate(np.concatenate([[0.0], c]))
    c[-1] = TOTAL
    return c.astype(np.uint32)


def adversarial_logits(rng, v, m):
    """(the generator of test_gpu_parity._adversarial_logits) columns that exercise ties, huge dynamic range, -inf, masses around
    2^-30 and f64 rounding of tiny terms"""
    cols = []
    cols.append(np.zeros(v, np.float32))                                   # all equal
    a = rng.normal(0, 1, v).astype(np.float32); a[v // 3] = 60.0; cols.append(a)   # one dominant symbol
    a = rng.normal(0, 12, v).astype(np.float32); cols.append(a)           # many terms far below ulp(sum)
    a = np.full(v, -np.inf, np.float32); a[5] = 0.0; a[v - 1] = -1.0; cols.append(a)  # -inf entries
    a = np.linspace(-25, 0, v).astype(np.float32); cols.append(a)          # masses straddling 2^-30
    a = np.full(v, -20.794415, np.float32); a[0] = 0.0; cols.append(a)      # e ~ 2^-30 each
    a = np.repeat(rng.normal(0, 3, v // 2 + 1).astype(np.float32), 2)[:v]; cols.append(a)  # exact ties
    a = (rng.normal(0, 40, v)).astype(np.float32); cols.append(a)          # underflow to exactly 0 for most entries
    while len(cols) < m:
        cols.append(rng.normal(0, rng.uniform(0.2, 8), v).astype(np.float32))
    return np.stack(cols[:m], axis=1)  # [V, M]


def encode_loop(session, ids, context=512, reprime_interval=512):
    """the reference's SmolLM encode loop (src/main.rs:1913-1916, 1935, 1979, 2275-2300, 2344-2358, as oracle/cz_loop.c restates it)
    coding with the floored alphabet; ids[0] is BOS.  Returns the payload."""
    eff = min(context, 511)
    logits = session.step_logits(ids[0])
    bounds = []
    for i in range(len(ids) - 1):
        sym = int(ids[i + 1])
        if session.index_pos() >= eff and i % reprime_interval == 0 and i > 0:
            end = 1 + i
            logits = session.reprime(ids[max(0, end - eff):end])
        cdf = cdf_floor(logits)
        bounds.append((int(cdf[sym]), int(cdf[sym + 1])))
        logits = session.step_logits(sym)
    return oracle.ac_encode(bounds)


def decode_loop(session, payload, bos, token_count, context=512, reprime_interval=512):
    """the reference's SmolLM decode loop (src/main.rs:2485-2654) with the floored alphabet; returns BOS + the decoded ids"""
    eff = min(context - 1, 511)
    dec = oracle.Decoder(payload)
    logits = session.step_logits(bos)
    out = [bos]
    for i in range(token_count):
        if session.index_pos() >= eff and i % reprime_interval == 0 and i > 0:
            end = len(out)
            logits = session.reprime(np.asarray(out[max(0, end - eff):end], np.uint32))
        sym = int(dec.decode(cdf_floor(logits)))
        out.append(sym)
        logits = session.step_logits(sym)
    return np.asarray(out, np.uint32)


def test_oracle_floor_cdf_equals_the_numpy_restatement_and_has_no_empty_interval():
    rng = np.random.default_rng(7)
    for v in (1024, 4099):
        logits = adversarial_logits(rng, v, 12)
        logits[:, 11] = rng.normal(0, 30, v)  # most entries more than 87 below the max
        for j in range(logits.shape[1]):
            cdf = cdf_floor(logits[:, j])
            assert np.array_equal(cdf, cdf_floor_numpy(logits[:, j])), (v, j)
            assert cdf[0] == 0 and cdf[-1] == TOTAL and np.all(np.diff(cdf.astype(np.int64)) >= 1), (v, j)
            # the unfloored alphabet has empty intervals on these columns; the floored one never does
            if j in (3, 7):
                assert np.any(np.diff(oracle.logits_to_cdf(logits[:, j], 0).astype(np.int64)) == 0), j


def _peaky_oracle():
    import candlezip_b200 as cz

    host = cz.Context(-1)
    m = cz.Model(host, cz.SMOLLM_TINY).random_init(5, 0.05, 1.5)  # the peaky model of the STORED fallback test
    cfg = dict(cz.SMOLLM_TINY, rms_eps=1e-5)
    return oracle.Session.llama(cfg, m.tensors())


def test_peaky_model_round_trips_on_the_oracle_loop_with_the_floor():
    """the model whose random-byte input hits a zero-width interval in the reference's (unfloored) loop codes and decodes that
    input with the floored alphabet, across a reprime"""
    ids = np.concatenate([[0], np.random.default_rng(0).integers(0, 256, 700)]).astype(np.uint32)
    with pytest.raises(ValueError, match="rc=-1"):  # -1: a zero-width interval
        _peaky_oracle().encode_tokens(ids)
    payload = encode_loop(_peaky_oracle(), ids)
    assert np.array_equal(decode_loop(_peaky_oracle(), payload, 0, len(ids) - 1), ids)


class _StubModel:
    """what decompress needs of a model when the container is rejected before any decoding, or to see what it was asked to decode"""

    def __init__(self, arch, ids=None):
        self.cfg = dict(arch=arch, vocab=1024)
        self.ids, self.calls = ids, []

    def decode(self, pays, seg, **kw):
        self.calls.append(kw)
        return self.ids


def test_pdf_floor_container_flag_writes_parses_and_is_validated():
    from candlezip_b200 import _lib, codec, container

    assert _lib.CZ_FLAG_PDF_FLOOR == 1 << 10
    data = bytes(range(40))
    ids = np.frombuffer(data, np.uint8).astype(np.uint32)
    f = dict(token_count=len(data), orig_len_bytes=len(data), vocab_size=1024, orig_hash16=container.blake3_16(data),
             reserved_flags=_lib.CZ_FLAG_PDF_FLOOR)
    pays = [b"\x12\x34", b"\x56"]
    blob = container.write_container(f, b"model.safetensors", pays, seg_tokens=[30, 10])
    g, _, _, _, st, p2 = container.read_container(blob)
    assert g["reserved_flags"] == _lib.CZ_FLAG_PDF_FLOOR | _lib.CZ_FLAG_SEGMENTS and list(st) == [30, 10] and p2 == pays
    # honoured: the payload is decoded with the floored alphabet
    smol = _StubModel(0, ids)
    assert codec.decompress(smol, blob) == data and smol.calls[-1]["pdf_floor"] is True
    plain = container.write_container(dict(f, reserved_flags=0), b"model.safetensors", pays, seg_tokens=[30, 10])
    assert codec.decompress(smol, plain) == data and smol.calls[-1]["pdf_floor"] is False
    # rejected: on RWKV-7 (its alphabet is floored already) and together with STORED
    with pytest.raises(ValueError, match="PDF_FLOOR"):
        codec.decompress(_StubModel(1, ids), blob)
    stored = container.write_container(dict(f, reserved_flags=_lib.CZ_FLAG_PDF_FLOOR | _lib.CZ_FLAG_STORED), b"model.safetensors", [data])
    with pytest.raises(ValueError, match="PDF_FLOOR"):
        codec.decompress(_StubModel(0, ids), stored)


def test_pdf_floor_options_are_validated_on_the_host():
    import candlezip_b200 as cz
    from candlezip_b200 import __main__ as cli
    from candlezip_b200 import _lib, codec

    with pytest.raises(ValueError, match="on_zero_width"):
        codec.compress(_StubModel(0), b"abc", on_zero_width="skip")
    with pytest.raises(SystemExit) as e:
        cli.main(["compress", "in.txt", "--reuse-scan-dir", "run", "--on-zero-width", "floor"])
    assert e.value.code == 2
    with pytest.raises(SystemExit):
        cli.main(["compress", "in.txt", "--on-zero-width", "never"])
    # the model-level switch: SmolLM takes it, RWKV-7 refuses (no device needed)
    import sys

    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from rwkv7_weights import RWKV7_TINY

    host = cz.Context(-1)
    sm = cz.Model(host, cz.SMOLLM_TINY)
    sm.set_pdf_floor(True)
    sm.set_pdf_floor(False)
    rm = cz.Model(host, RWKV7_TINY)
    rm.set_pdf_floor(False)
    with pytest.raises(cz.CzError) as err:
        rm.set_pdf_floor(True)
    assert err.value.code == _lib.CZ_ERR_UNSUPPORTED
    assert _lib.lib.cz_model_set_pdf_floor(None, 1) == _lib.CZ_ERR_INVALID
