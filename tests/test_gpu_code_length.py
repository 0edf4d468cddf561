"""GPU suite for per-token code lengths: the coding-distribution entropy kernel (cz_cdf_entropy) against a numpy reference over the
oracle's CDFs, the encode-side sinks (cz_model_set_code_length_out) on both architectures against the oracle CDF of the same logits,
their invariance, the coder's accounting, zero-width tokens, and the `analyze` command."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
from candlezip_b200 import _lib, codec
from test_cpu_pdf_floor import adversarial_logits, cdf_floor

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
TOL = 1e-12


def entropy_ref(cdf):
    """2^-30 sum_{w_s > 0} w_s (30 - log2 w_s) over the widths of a quantised CDF, added in ascending s.  30 - log2 w is evaluated as
    -log2(1 - (2^30 - w) 2^-30) through log1p where it is below 1 (w > 2^29): there the plain form loses digits to cancellation."""
    w = np.diff(np.asarray(cdf, np.int64))
    w = w[w > 0]
    big = w > (1 << 29)
    bits = np.where(big, -np.log1p(-((1 << 30) - w) * 2.0 ** -30) / np.log(2.0), 30.0 - np.log2(w.astype(np.float64)))
    return float(np.add.accumulate(w * bits)[-1]) * 2.0 ** -30


def oracle_cdf(col, mode):
    return cdf_floor(col) if mode == _lib.CZ_CDF_SMOLLM_FLOOR else oracle.logits_to_cdf(col, mode)


def _close(got, want):
    return abs(got - want) <= TOL * max(abs(want), 1e-300)


@pytest.mark.parametrize("v,mode", [(1024, 0), (1024, 2), (4099, 0), (4099, 2), (49152, 0), (49152, 2), (65536, 1), (1024, 1)])
def test_entropy_kernel_against_reference(gpu_ctx, v, mode):
    """random columns, peaky ones with zero-width symbols, all-equal ones, -inf entries; 40 and 1,027 columns go through the direct-load
    stats kernel, 260 and 1,024 through the TMA-staged one: every column's H within 1e-12 of the reference, and bit-identical whichever
    batch it is in"""
    rng = np.random.default_rng(v + 7 * mode)
    big = adversarial_logits(rng, v, 1027)
    big[:, 8] = rng.normal(0, 30, v)  # mostly far below the max: the fast expf's fallback, many zero widths
    big[:, 9] = 0.0
    big[3, 9] = 80.0  # one symbol with all the mass: every other width is 0 (or 1 under the floor)
    want = {}
    first = None
    for m in (40, 260, 1027, 1024):
        lg = np.ascontiguousarray(big[:, :m])
        h = gpu_ctx.cdf_entropy(lg, mode)
        assert h.shape == (m,) and np.all(np.isfinite(h)) and np.all(h >= 0)
        cols = range(m) if m <= 260 or v <= 4099 else list(range(64)) + list(rng.choice(m, 96, replace=False))
        for j in cols:
            if j not in want:
                want[j] = entropy_ref(oracle_cdf(lg[:, j], mode))
            assert _close(h[j], want[j]), (v, mode, m, j, h[j], want[j])
        if first is None:
            first = h[:40].copy()
        assert np.array_equal(h[:40].view(np.uint64), first.view(np.uint64)), (v, mode, m)
    # the all-equal column: the widths of a uniform quantisation
    c0 = oracle_cdf(big[:, 0], mode)
    assert _close(first[0], entropy_ref(c0))
    # a few columns against cz_cdf_full's widths
    for j in (0, 1, 5, 8, 9, 17):
        full = gpu_ctx.cdf_full(big[:, j], mode)
        assert np.array_equal(full, oracle_cdf(big[:, j], mode)), j
        assert _close(first[j], entropy_ref(full)), j


def test_entropy_kernel_arguments(gpu_ctx):
    """mode 0 falls back to the uniform pdf only when S <= 0, which a column cannot produce (its maximum's own term is 1; a column
    without a maximum, all NaN or all -inf, is NaN and refused like cz_cdf_bounds refuses it); unknown modes and bad shapes are refused"""
    lg = np.zeros((64, 4), np.float32)
    h = gpu_ctx.cdf_entropy(lg, 0)
    assert np.allclose(h, 6.0, rtol=1e-15, atol=0)  # 64 equal widths of 2^24: log2 64
    bad = lg.copy()
    bad[:, 2] = -np.inf
    with pytest.raises(cz.CzError) as e:
        gpu_ctx.cdf_entropy(bad, 0)
    assert e.value.code == _lib.CZ_ERR_INVALID
    for mode in (3, -1):
        with pytest.raises(cz.CzError) as e:
            gpu_ctx.cdf_entropy(lg, mode)
        assert e.value.code == _lib.CZ_ERR_INVALID
    out = np.zeros(4)
    assert _lib.lib.cz_cdf_entropy(gpu_ctx._h, lg.ctypes.data_as(_lib.f32p), 64, 4, 3, 0, out.ctypes.data_as(_lib.f64p)) == _lib.CZ_ERR_INVALID
    assert _lib.lib.cz_cdf_entropy(gpu_ctx._h, lg.ctypes.data_as(_lib.f32p), 64, 4, 4, 0, None) == _lib.CZ_ERR_INVALID
    assert _lib.lib.cz_cdf_entropy(gpu_ctx._h, lg.ctypes.data_as(_lib.f32p), 0, 4, 4, 0, out.ctypes.data_as(_lib.f64p)) == _lib.CZ_ERR_INVALID
    one = gpu_ctx.cdf_entropy(np.zeros((1, 3), np.float32), 0)
    assert np.array_equal(one, np.zeros(3))  # a one-symbol alphabet: the whole interval, 0 bits


def _rwkv_tiny(gpu_ctx):
    from rwkv7_weights import RWKV7_TINY, make_weights

    model = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        model.set_tensor(name, arr)
    return model


def _chunks(n, reprime):
    return list(zip(*codec.schedule_chunks(n, 512, 512))) if reprime else [(0, n)]


def _check_against_chunk_logits(gpu_ctx, model, ids, r, mode, reprime, segs=None):
    """every token of the checked segments: the interval is (cdf[s], cdf[s+1]) of the oracle CDF of the GPU's teacher-forced logits for
    its chunk, and the entropy is cz_cdf_entropy of those logits, bit for bit, and the reference entropy of that CDF within 1e-12"""
    seg_start = r["seg_start"]
    for g in segs if segs is not None else range(len(seg_start) - 1):
        a, b = int(seg_start[g]), int(seg_start[g + 1])
        seq = np.concatenate([[0], ids[a:b]]).astype(np.uint32)
        for f, k in _chunks(b - a, reprime):
            f, k = int(f), int(k)
            p0 = 0 if f == 0 else f + 1 - min(f + 1, 511)
            lg = model.chunk_logits(seq[p0:f + 1], ids[a + f:a + f + k])
            ent = gpu_ctx.cdf_entropy(np.ascontiguousarray(lg.T), mode)
            assert np.array_equal(ent.view(np.uint64), r["entropy"][a + f:a + f + k].view(np.uint64)), (g, f)
            for j in range(k):
                cdf = oracle_cdf(lg[j], mode)
                s = int(ids[a + f + j])
                assert (int(r["c_lo"][a + f + j]), int(r["c_hi"][a + f + j])) == (int(cdf[s]), int(cdf[s + 1])), (g, f, j)
                assert _close(r["entropy"][a + f + j], entropy_ref(cdf)), (g, f, j, r["entropy"][a + f + j])


def _check_accounting(r):
    """per segment: sum bits - 32 <= 8 len(payload) <= sum bits + sum log2(w / (w - 1)) + 9"""
    w = r["c_hi"].astype(np.int64) - r["c_lo"].astype(np.int64)
    with np.errstate(divide="ignore"):
        loss = np.log2(w / (w - 1.0))
    for g, pay in enumerate(r["payloads"]):
        a, b = int(r["seg_start"][g]), int(r["seg_start"][g + 1])
        bits = float(np.sum(r["bits"][a:b]))
        assert bits - 32 <= 8 * len(pay) <= bits + float(np.sum(loss[a:b])) + 9, (g, bits, 8 * len(pay))


def _plain_launches(model, ids, **kw):
    n0 = model.ctx.launch_count()
    pays = model.encode(ids, **kw)[0]
    return pays, model.ctx.launch_count() - n0


@pytest.mark.parametrize("arch", ["smollm", "rwkv7"])
def test_encode_sinks(gpu_ctx, arch):
    if arch == "smollm":
        model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 0.05)
        V, mode, reprime = 1024, 0, True
        ids = np.random.default_rng(3).integers(0, V, 1900).astype(np.uint32)
    else:
        model = _rwkv_tiny(gpu_ctx)
        V, mode, reprime = model.cfg["vocab"], 1, False
        rng = np.random.default_rng(4)
        ids = rng.integers(0, V, 900).astype(np.uint32)
        mask = rng.random(900) < 0.1
        ids[mask] = V + rng.integers(0, 256, int(mask.sum()))  # literal escapes
    pays, plain = _plain_launches(model, ids, n_segments=3)
    # all sinks off (set and cleared): the same launches, the same bytes
    h = model._h
    lo = np.zeros(len(ids), np.uint32)
    _lib.check(_lib.lib.cz_model_set_code_length_out(h, lo.ctypes.data_as(_lib.u32p), None, None, len(ids)))
    _lib.check(_lib.lib.cz_model_set_code_length_out(h, None, None, None, 0))
    again, n_off = _plain_launches(model, ids, n_segments=3)
    assert again == pays and n_off == plain
    n0 = gpu_ctx.launch_count()
    r = model.analyze(ids, n_segments=3)
    assert gpu_ctx.launch_count() - n0 > plain
    assert np.all(np.isfinite(r["entropy"])) and np.all(r["entropy"] >= 0)
    assert r["payloads"] == pays and np.all(r["first_zw"] == np.uint64(_lib.NO_ZERO_WIDTH))
    assert np.array_equal(r["bits"], 30.0 - np.log2((r["c_hi"].astype(np.int64) - r["c_lo"]).astype(np.float64)))
    _check_against_chunk_logits(gpu_ctx, model, ids, r, mode, reprime)
    _check_accounting(r)
    # invariance: wave / slab size and segment split change neither the intervals nor the entropies of a token
    for kw in (dict(max_batch_tokens=700), dict(max_batch_tokens=257)):
        r2 = model.analyze(ids, n_segments=3, **kw)
        assert r2["payloads"] == pays
        for k in ("c_lo", "c_hi", "entropy"):
            assert np.array_equal(r2[k].view(np.uint8), r[k].view(np.uint8)), (kw, k)
    for g in range(3):
        a, b = int(r["seg_start"][g]), int(r["seg_start"][g + 1])
        r3 = model.analyze(ids[a:b])
        assert r3["payloads"] == [pays[g]]
        for k in ("c_lo", "c_hi", "entropy"):
            assert np.array_equal(r3[k].view(np.uint8), r[k][a:b].view(np.uint8)), (g, k)
    # the sinks were cleared: a plain encode launches what it did before
    assert _plain_launches(model, ids, n_segments=3) == (pays, plain)
    # a sink smaller than the call is refused, and nothing is written
    small = np.full(len(ids) - 1, 7, np.uint32)
    _lib.check(_lib.lib.cz_model_set_code_length_out(h, small.ctypes.data_as(_lib.u32p), None, None, small.shape[0]))
    try:
        with pytest.raises(cz.CzError) as e:
            model.encode(ids, n_segments=3)
        assert e.value.code == _lib.CZ_ERR_INVALID and np.all(small == 7)
    finally:
        _lib.check(_lib.lib.cz_model_set_code_length_out(h, None, None, None, 0))
    model.close()


def test_full_size_smollm_sinks(gpu_ctx):
    """SmolLM-135M shape (V = 49,152, the TMA stats kernel and the e-cache), 1,300 tokens in 2 segments: segment 0's intervals and
    entropies (a chunk of 512 and a reprimed one) against the oracle CDF and cz_cdf_entropy of the same logits"""
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(5, 0.02, 0.02)
    ids = np.random.default_rng(23).integers(0, 49152, 1300).astype(np.uint32)
    r = model.analyze(ids, n_segments=2)
    assert r["payloads"] == model.encode(ids, n_segments=2)[0]
    _check_against_chunk_logits(gpu_ctx, model, ids, r, 0, True, segs=[0])
    _check_accounting(r)
    model.close()


def test_zero_width_tokens_and_floor(gpu_ctx):
    """the peaky tiny model (random tokens are zero-width unfloored): unfloored analysis reports +inf exactly at the zero-width tokens,
    the first of each segment being the one first_zw names; floored analysis reports none and its intervals and entropies are mode 2's"""
    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 1.5)
    ids = np.random.default_rng(9).integers(0, 1024, 1700).astype(np.uint32)
    r = model.analyze(ids, n_segments=3)
    inf = ~np.isfinite(r["bits"])
    assert inf.any() and np.array_equal(inf, r["c_lo"] == r["c_hi"]) and np.all(r["bits"][inf] == np.inf)
    assert np.all(np.isfinite(r["entropy"])) and np.all(r["entropy"] >= 0)  # (zero widths between non-zero ones add nothing)
    for g in range(3):
        a, b = int(r["seg_start"][g]), int(r["seg_start"][g + 1])
        zi = np.nonzero(inf[a:b])[0]
        assert int(r["first_zw"][g]) == (int(zi[0]) if zi.size else _lib.NO_ZERO_WIDTH), g
    _check_against_chunk_logits(gpu_ctx, model, ids, r, 0, True, segs=[0])
    rf = model.analyze(ids, n_segments=3, pdf_floor=True)
    assert np.all(np.isfinite(rf["bits"])) and np.all(rf["first_zw"] == np.uint64(_lib.NO_ZERO_WIDTH))
    assert rf["payloads"] == model.encode(ids, n_segments=3, pdf_floor=True)[0]
    _check_against_chunk_logits(gpu_ctx, model, ids, rf, _lib.CZ_CDF_SMOLLM_FLOOR, True, segs=[1])
    _check_accounting(rf)
    assert not np.array_equal(rf["entropy"], r["entropy"])
    model.close()


@pytest.mark.parametrize("backend,size,segments", [("smollm", 65536, 4), ("rwkv7", 8192, 2)])
def test_cli_analyze(tmp_path, backend, size, segments):
    """`analyze` on an enwik8 stand-in slice writes an npz whose summary matches its arrays"""
    import corpus

    src = tmp_path / "enwik8_slice"
    data = corpus.load("enwik8_3mib")[:size]
    src.write_bytes(data)
    out = tmp_path / "slice.npz"
    r = subprocess.run([sys.executable, "-m", "candlezip_b200", "analyze", str(src), str(out), "--backend", backend, "--segments", str(segments)],
                       cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, (r.stdout, r.stderr[-2000:])
    z = np.load(out)
    s = json.loads(str(z["summary"]))
    bits = z["bits"]
    fin = np.isfinite(bits)
    assert s["tokens"] == len(z["ids"]) == len(data) and s["bytes"] == len(data)
    assert abs(s["bits"] - float(bits[fin].sum())) <= 1e-9 * s["bits"]
    assert s["payload_bits"] == 8 * int(z["payload_lens"].sum())
    assert abs(s["mean_entropy"] - float(z["entropy"].mean())) <= 1e-12 * s["mean_entropy"]
    assert s["zero_width"] == int((~fin).sum()) and len(s["segments"]) == segments
    assert [seg["tokens"] for seg in s["segments"]] == np.diff(z["seg_start"].astype(np.int64)).tolist()
    assert sum(b["tokens"] for b in s["by_chunk_position"]) == s["tokens"] == sum(b["tokens"] for b in s["by_segment_position"])
    assert np.array_equal(z["segment_position"], np.concatenate([np.arange(n) for n in np.diff(z["seg_start"].astype(np.int64))]))
    assert s == codec.summarize(bits, z["entropy"], z["segment"], z["segment_position"], z["chunk_position"], z["payload_lens"], len(data))
    assert "wrote" in r.stdout and "zero-width" in r.stdout
    if backend == "smollm":
        assert z["chunk"].max() >= 1  # 16 KiB segments are reprimed
    else:
        assert not z["chunk"].any()
