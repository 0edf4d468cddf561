"""GPU suite (-m gpu): the CUDA path, through the C ABI, against the oracle on the same seeded inputs.
Bit-exact for integer/byte work (CDF bounds, symbols, bitstreams, tokens); stated tolerances for logits."""
import ctypes as C
import os

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
from candlezip_b200 import _lib

pytestmark = pytest.mark.gpu
TOTAL = 1 << 30


def _adversarial_logits(rng, v, m):
    """columns that exercise ties, huge dynamic range, -inf, masses around 2^-30 and f64 rounding of tiny terms"""
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


@pytest.mark.parametrize("v,m", [(1024, 8), (4099, 37), (49152, 40)])
def test_k1_cdf_bounds_bit_exact(gpu_ctx, v, m):
    rng = np.random.default_rng(v + m)
    logits = _adversarial_logits(rng, v, m)
    syms = rng.integers(0, v, m).astype(np.uint32)
    syms[:4] = [0, v - 1, 1, v - 2]
    lo, hi = gpu_ctx.cdf_bounds(logits, syms)
    for j in range(m):
        cdf = oracle.logits_to_cdf(logits[:, j], 0)
        assert (int(lo[j]), int(hi[j])) == (int(cdf[syms[j]]), int(cdf[syms[j] + 1])), (j, syms[j])


def test_k1_cdf_full_bit_exact(gpu_ctx):
    rng = np.random.default_rng(0)
    for v in (257, 5000):
        logits = rng.normal(0, 6, v).astype(np.float32)
        for mode in (0, 1):
            assert np.array_equal(gpu_ctx.cdf_full(logits, mode), oracle.logits_to_cdf(logits, mode)), (v, mode)


@pytest.mark.parametrize("mode", [0, 1])
def test_k1_cdf_search_bit_exact(gpu_ctx, mode):
    rng = np.random.default_rng(11 + mode)
    v, m = 3000, 70
    logits = _adversarial_logits(rng, v, m)
    values = rng.integers(0, TOTAL, m).astype(np.uint32)
    values[:3] = [0, TOTAL - 1, 1]
    sym, lo, hi = gpu_ctx.cdf_search(logits, values, mode)
    for j in range(m):
        cdf = oracle.logits_to_cdf(logits[:, j], mode)
        s = int(np.searchsorted(cdf, values[j], side="right") - 1)
        assert (int(sym[j]), int(lo[j]), int(hi[j])) == (s, int(cdf[s]), int(cdf[s + 1])), j


def test_k1_rwkv_literal_mode_bounds(gpu_ctx):
    rng = np.random.default_rng(5)
    v, m = 2048, 33
    logits = _adversarial_logits(rng, v, m)
    syms = rng.integers(0, v + 256, m).astype(np.uint32)
    syms[:3] = [v, v + 255, v - 1]
    lo, hi = gpu_ctx.cdf_bounds(logits, syms, mode=1)
    for j in range(m):
        cdf = oracle.logits_to_cdf(logits[:, j], 1)
        assert (int(lo[j]), int(hi[j])) == (int(cdf[syms[j]]), int(cdf[syms[j] + 1])), j
        assert hi[j] > lo[j]  # the floor guarantees a non-empty interval


@pytest.mark.parametrize("mode", [0, 1])
def test_k9_xe_bits(gpu_ctx, mode):
    rng = np.random.default_rng(2)
    v, m = 1500, 20
    logits = rng.normal(0, 5, (v, m)).astype(np.float32)
    syms = rng.integers(0, v, m).astype(np.uint32)
    got = gpu_ctx.xe_bits_cols(logits, syms, mode)
    for j in range(m):
        pdf = oracle.combined_pdf_with_literals(logits[:, j]) if mode else oracle.softmax_pdf_floor(logits[:, j])
        want = -np.log2(max(pdf[syms[j]], 1e-300))
        assert abs(got[j] - want) <= 1e-12 * max(1.0, abs(want)), j  # f64; only log2's last ulp may differ


def test_k2_encoder_lanes_bit_exact(gpu_ctx):
    rng = np.random.default_rng(3)
    lanes, bounds_all, off = [], [], [0]
    for lane in range(41):
        n = int(rng.integers(0, 400)) if lane else 0  # lane 0 is the empty stream -> 0x40
        b = []
        for _ in range(n):
            kind = rng.integers(0, 4)
            if kind == 0:
                lo = int(rng.integers(0, TOTAL - 1)); hi = lo + 1          # narrowest interval: long carry runs
            elif kind == 1:
                lo = int(rng.integers(0, TOTAL // 2)); hi = int(rng.integers(lo + 1, TOTAL + 1))
            elif kind == 2:
                lo = (TOTAL // 2) - int(rng.integers(1, 5)); hi = (TOTAL // 2) + int(rng.integers(1, 5))  # straddles 1/2 (E3)
            else:
                lo, hi = 0, TOTAL                                         # probability-1 symbol: no bits
            b.append((lo, hi))
        lanes.append(b)
        bounds_all += b
        off.append(len(bounds_all))
    lo = np.array([b[0] for b in bounds_all], np.uint32)
    hi = np.array([b[1] for b in bounds_all], np.uint32)
    got = gpu_ctx.ac_encode_lanes(lo, hi, off)
    for lane, b in enumerate(lanes):
        assert got[lane] == oracle.ac_encode(b), lane
    assert got[0] == bytes([0x40])


def test_k2_zero_width_is_an_error(gpu_ctx):
    with pytest.raises(cz.CzError) as e:
        gpu_ctx.ac_encode_lanes([1, 7], [2, 7], [0, 2])
    assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH


def test_k3_decoder_lanes_roundtrip(gpu_ctx):
    rng = np.random.default_rng(4)
    w = rng.integers(1, 1000, 300).astype(np.float64)
    cdf = np.concatenate([[0], np.floor(np.cumsum(w) / w.sum() * TOTAL)]).astype(np.uint32)
    cdf[-1] = TOTAL
    off, syms_all, pays = [0], [], []
    for lane in range(23):
        n = int(rng.integers(1, 500))
        syms = rng.integers(0, 300, n)
        pays.append(oracle.ac_encode([(int(cdf[s]), int(cdf[s + 1])) for s in syms]))
        syms_all += list(syms)
        off.append(len(syms_all))
    got = gpu_ctx.ac_decode_lanes(pays, off, cdf)
    assert np.array_equal(got, np.array(syms_all, np.uint32))


# ------------------------------------------------------------------ dense contraction engines
def _bf16(a):
    a = np.ascontiguousarray(a, np.float32)
    u = a.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return u.astype(np.uint16)


def _bf16_to_f32(b):
    return (b.astype(np.uint32) << 16).view(np.float32)


def _run_gemm(ctx, engine, a16, b16, epi, bn, c_init, ldc):
    M, K = a16.shape
    N = b16.shape[0]
    c = np.ascontiguousarray(c_init).copy()
    _lib.check(_lib.lib.cz_test_gemm(ctx._h, engine, M, N, K, a16.ctypes.data_as(C.POINTER(C.c_uint16)),
                                     b16.ctypes.data_as(C.POINTER(C.c_uint16)), epi, bn, c.ctypes.data_as(C.c_void_p), ldc))
    return c


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
@pytest.mark.parametrize("M,N,K,bn", [(128, 192, 64, 192), (300, 960, 576, 192), (1000, 576, 1536, 192), (49152 // 8, 77, 576, 256),
                                      (129, 200, 192, 192)])
def test_gemm_store_f32(gpu_ctx, engine, M, N, K, bn):
    rng = np.random.default_rng(M + N + K)
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    b16 = _bf16(rng.normal(0, 1, (N, K)))
    ldc = (N + 3) // 4 * 4
    c = _run_gemm(gpu_ctx, engine, a16, b16, 0, bn, np.zeros((M, ldc), np.float32), ldc)
    want = _bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T
    err = np.abs(c[:, :N] - want).max()
    assert err < 2e-3 * np.sqrt(K / 64), (err,)
    assert np.all(c[:, N:] == 0)


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
def test_gemm_epilogues(gpu_ctx, engine):
    rng = np.random.default_rng(8)
    M, K, F = 260, 192, 576
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    # residual add
    b16 = _bf16(rng.normal(0, 0.2, (192, K)))
    base = rng.normal(0, 1, (M, 192)).astype(np.float32)
    c = _run_gemm(gpu_ctx, engine, a16, b16, 1, 192, base, 192)
    want = base + _bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T
    assert np.abs(c - want).max() < 5e-3
    # swiglu over packed gate/up rows (groups of 96)
    wg = _bf16(rng.normal(0, 0.1, (F, K)))
    wu = _bf16(rng.normal(0, 0.1, (F, K)))
    packed = np.empty((2 * F, K), np.uint16)
    for g in range(F // 96):
        packed[g * 192 : g * 192 + 96] = wg[g * 96 : (g + 1) * 96]
        packed[g * 192 + 96 : (g + 1) * 192] = wu[g * 96 : (g + 1) * 96]
    out16 = _run_gemm(gpu_ctx, engine, a16, packed, 2, 192, np.zeros((M, F), np.uint16), F)
    A = _bf16_to_f32(a16).astype(np.float64)
    gate = A @ _bf16_to_f32(wg).astype(np.float64).T
    up = A @ _bf16_to_f32(wu).astype(np.float64).T
    want = gate / (1 + np.exp(-gate)) * up
    got = _bf16_to_f32(out16)
    assert np.abs(got - want).max() < 0.02 * max(1.0, np.abs(want).max())
    # bf16 store
    o16 = _run_gemm(gpu_ctx, engine, a16, b16, 3, 192, np.zeros((M, 192), np.uint16), 192)
    want = A @ _bf16_to_f32(b16).astype(np.float64).T
    assert np.abs(_bf16_to_f32(o16) - want).max() < 0.02 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
@pytest.mark.parametrize("epi,bn,fn", [(5, 192, np.tanh), (6, 192, lambda x: 1 / (1 + np.exp(-x))), (7, 256, lambda x: np.maximum(x, 0) ** 2)],
                         ids=["tanh", "sigmoid", "relusq"])
def test_gemm_activation_epilogues(gpu_ctx, engine, epi, bn, fn):
    """RWKV-7 LoRA / FFN epilogues (rwkv7.rs:212, 234, 426), incl. a ragged N (tail columns stay untouched)."""
    rng = np.random.default_rng(epi)
    M, K, N = 333, 128, 200
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    b16 = _bf16(rng.normal(0, 0.15, (N, K)))
    ldc = 208
    out = _run_gemm(gpu_ctx, engine, a16, b16, epi, bn, np.full((M, ldc), 0x7FC0, np.uint16), ldc)
    want = fn(_bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T)
    assert np.abs(_bf16_to_f32(out[:, :N]) - want).max() < 0.01 * max(1.0, np.abs(want).max())
    assert np.all(out[:, N:] == 0x7FC0)


@pytest.mark.parametrize("epi", [0, 4], ids=["store", "colmax"])
def test_gemm_tma_store_many_tiles_few_columns(gpu_ctx, epi):
    """decode-shaped LM head: thousands of vocab rows (many M tiles per CTA), a handful of columns.  Every tile then stores
    through the same 32-column chunk: regression test for the double-buffered TMA patch being alternated per chunk index
    instead of per store (consecutive tiles overwrote a patch that a bulk store was still reading)."""
    rng = np.random.default_rng(40 + epi)
    M, N, K = 128 * 148 * 3 + 77, 3, 128
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    b16 = _bf16(rng.normal(0, 1, (N, K)))
    c = _run_gemm(gpu_ctx, _lib.CZ_ENGINE_TCGEN05, a16, b16, epi, 256, np.zeros((M, 4), np.float32), 4)
    want = _bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T
    assert np.abs(c[:, :N] - want).max() < 5e-3
    assert np.all(c[:, N:] == 0)


def test_gemm_lm_head_grouped_raster(gpu_ctx):
    """More column tiles than CTAs: the LM-head GEMM walks the column tiles in L2-sized groups (every vocabulary tile of a group
    before the next group, the last group partial); every output element must still be written exactly once."""
    rng = np.random.default_rng(77)
    M, N, K = 300, 157 * 256 - 40, 64
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    b16 = _bf16(rng.normal(0, 1, (N, K)))
    ldc = (N + 3) // 4 * 4
    c = _run_gemm(gpu_ctx, _lib.CZ_ENGINE_TCGEN05, a16, b16, 4, 256, np.full((M, ldc), -7.0, np.float32), ldc)
    want = _bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T
    assert np.abs(c[:, :N] - want).max() < 2e-3


def test_gemm_tcgen05_row_invariance(gpu_ctx):
    """decode safety: a row's result must not depend on batch size or on its position in the tile grid."""
    rng = np.random.default_rng(12)
    K, N = 576, 960
    b16 = _bf16(rng.normal(0, 1, (N, K)))
    rows = _bf16(rng.normal(0, 1, (700, K)))
    big = _run_gemm(gpu_ctx, _lib.CZ_ENGINE_TCGEN05, rows, b16, 0, 192, np.zeros((700, N), np.float32), N)
    for sel in ([0], [5, 131, 699], list(range(257, 300))):
        small = _run_gemm(gpu_ctx, _lib.CZ_ENGINE_TCGEN05, np.ascontiguousarray(rows[sel]), b16, 0, 192, np.zeros((len(sel), N), np.float32), N)
        assert np.array_equal(small.view(np.uint32), big[sel].view(np.uint32)), sel


def _run_gemm_norm(ctx, a16, b16, b2_16, w_next, eps, x):
    M, K = a16.shape
    N, N2 = b16.shape[0], b2_16.shape[0]
    x = np.ascontiguousarray(x, np.float32).copy()
    xb = np.zeros((M, N), np.uint16)
    ssq = np.zeros((M, (N // 192) * 3), np.float32)
    out2 = np.zeros((M, N2), np.uint16)
    u16p, f32p = C.POINTER(C.c_uint16), C.POINTER(C.c_float)
    w = np.ascontiguousarray(w_next, np.float32)
    _lib.check(_lib.lib.cz_test_gemm_norm(ctx._h, M, N, K, N2, a16.ctypes.data_as(u16p), b16.ctypes.data_as(u16p), b2_16.ctypes.data_as(u16p),
                                          w.ctypes.data_as(f32p), eps, x.ctypes.data_as(f32p), xb.ctypes.data_as(u16p),
                                          ssq.ctypes.data_as(f32p), out2.ctypes.data_as(u16p)))
    return x, xb, ssq, out2


@pytest.mark.parametrize("M", [1, 77, 300])
def test_gemm_fused_residual_rmsnorm(gpu_ctx, M):
    """EPI_ADD_NORM (residual add + bf16(x * w) + partial sums of squares) and the consumer's 1/rms row scale together equal
    residual add -> RMSNorm -> projection (LLaMA block structure, candle-transformers llama.rs reached from src/models.rs:94);
    rows are independent of the batch they are computed in (decode safety)."""
    rng = np.random.default_rng(40 + M)
    N, K, N2, eps = 576, 1536, 200, 1e-5
    a16 = _bf16(rng.normal(0, 1, (M, K)))
    b16 = _bf16(rng.normal(0, 0.05, (N, K)))
    b2 = _bf16(rng.normal(0, 0.1, (N2, N)))
    w = rng.uniform(0.5, 1.5, N).astype(np.float32)
    x0 = rng.normal(0, 1, (M, N)).astype(np.float32)
    x, xb, ssq, out2 = _run_gemm_norm(gpu_ctx, a16, b16, b2, w, eps, x0)
    want_x = x0.astype(np.float64) + _bf16_to_f32(a16).astype(np.float64) @ _bf16_to_f32(b16).astype(np.float64).T
    assert np.abs(x - want_x).max() < 5e-3
    # bf16(x * w) is exact given the device's own fp32 x
    assert np.array_equal(xb, _bf16(x * w))
    assert np.allclose(ssq.sum(1), (x.astype(np.float64) ** 2).sum(1), rtol=1e-5)
    rs = 1.0 / np.sqrt((x.astype(np.float64) ** 2).mean(1) + eps)
    want2 = (_bf16_to_f32(xb).astype(np.float64) @ _bf16_to_f32(b2).astype(np.float64).T) * rs[:, None]
    got2 = _bf16_to_f32(out2)
    assert np.abs(got2 - want2).max() < 2e-2 * max(1.0, np.abs(want2).max())
    if M >= 77:  # the same rows alone give the same bits
        sel = [0, 5, 76]
        xs, xbs, ssqs, out2s = _run_gemm_norm(gpu_ctx, np.ascontiguousarray(a16[sel]), b16, b2, w, eps, x0[sel])
        assert np.array_equal(xs.view(np.uint32), x[sel].view(np.uint32))
        assert np.array_equal(xbs, xb[sel]) and np.array_equal(ssqs.view(np.uint32), ssq[sel].view(np.uint32))
        assert np.array_equal(out2s, out2[sel])


# ------------------------------------------------------------------ SmolLM forward / encode / decode
def _tiny(gpu_ctx, engine, seed=5, embed_std=0.05):
    return cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(seed, 0.05, embed_std)


def _oracle_for(model, round_bf16):
    cfg = dict(model.cfg)
    cfg["rms_eps"] = cfg.pop("norm_eps")
    return oracle.Session.llama(cfg, model.tensors(), round_bf16=round_bf16)


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
def test_tiny_logits_vs_oracle(gpu_ctx, engine):
    model = _tiny(gpu_ctx, engine, embed_std=0.2)
    rng = np.random.default_rng(1)
    prime = rng.integers(0, 1024, 37).astype(np.uint32)
    targets = rng.integers(0, 1024, 9).astype(np.uint32)
    got = model.chunk_logits(prime, targets)
    orc = _oracle_for(model, round_bf16=1)
    ref = _oracle_for(model, round_bf16=0)
    want = [orc.reprime(prime)] + [orc.step_logits(t) for t in targets[:-1]]
    want32 = [ref.reprime(prime)] + [ref.step_logits(t) for t in targets[:-1]]
    for j in range(len(targets)):
        scale = max(1.0, np.abs(want32[j]).max())
        # vs the oracle with the same bf16 rounding points: only accumulation order differs
        assert np.abs(got[j] - want[j]).max() < 0.03 * scale, j
        # vs the reference's pure-f32 CPU semantics: the stated logits tolerance of the bf16 path
        assert np.abs(got[j] - want32[j]).max() < 0.06 * scale, j


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
def test_tiny_stepwise_equals_teacher_forced_bitwise(gpu_ctx, engine):
    model = _tiny(gpu_ctx, engine, embed_std=0.2)
    rng = np.random.default_rng(2)
    prime = rng.integers(0, 1024, 150).astype(np.uint32)
    targets = rng.integers(0, 1024, 140).astype(np.uint32)
    tf = model.chunk_logits(prime, targets)
    s = model.session()
    step = [s.reprime_with_history_and_get_last_logits_tensor(prime)]
    for t in targets[:-1]:
        step.append(s.step_logits_tensor(t))
    step = np.stack(step)
    assert np.array_equal(tf.view(np.uint32), step.view(np.uint32)), "teacher-forced and stepwise logits differ bitwise"
    assert s.index_pos() == len(prime) + len(targets) - 1


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
@pytest.mark.parametrize("n,n_seg", [(1, 1), (700, 1), (1700, 1), (2300, 3), (513, 5)])
def test_tiny_roundtrip_and_oracle_bitstream(gpu_ctx, engine, n, n_seg):
    model = _tiny(gpu_ctx, engine)
    rng = np.random.default_rng(n + n_seg)
    ids = rng.integers(0, 1024, n).astype(np.uint32)
    pays, seg_start = model.encode(ids, n_segments=n_seg)
    assert len(pays) == len(seg_start) - 1
    # (1) bitstream parity: GPU logits -> ORACLE quantiser + ORACLE coder must reproduce the GPU payload bit for bit
    g = 0
    a, b = int(seg_start[g]), int(seg_start[g + 1])
    seq = np.concatenate([[0], ids[a:b]]).astype(np.uint32)
    first = min(512, b - a)
    logits = model.chunk_logits([0], ids[a : a + first])
    bounds = [tuple(int(x) for x in oracle.logits_to_cdf(logits[j], 0)[[ids[a + j], ids[a + j] + 1]]) for j in range(first)]
    if b - a > 512:  # second chunk: prime = seq[2..513)
        second = min(512, b - a - 512)
        logits2 = model.chunk_logits(seq[2:513], ids[a + 512 : a + 512 + second])
        bounds += [tuple(int(x) for x in oracle.logits_to_cdf(logits2[j], 0)[[ids[a + 512 + j], ids[a + 512 + j] + 1]]) for j in range(second)]
    if len(bounds) == b - a:
        assert oracle.ac_encode(bounds) == pays[g]
    # (2) round trip through the batched lock-step decoder
    out = model.decode(pays, seg_start)
    assert np.array_equal(out, ids)
    # (3) compressed size vs the CPU oracle on the same weights (bits/byte parity, <= 0.5 %)
    if n >= 700 and n_seg == 1:
        orc = _oracle_for(model, round_bf16=0)
        ref_payload, _ = orc.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32))
        assert abs(len(pays[0]) - len(ref_payload)) <= 0.005 * len(ref_payload) + 2


def test_tiny_segment_invariance(gpu_ctx):
    """identical bytes whatever the wave size; per-segment streams equal single-stream encodes of the same tokens"""
    model = _tiny(gpu_ctx, _lib.CZ_ENGINE_TCGEN05)
    rng = np.random.default_rng(77)
    ids = rng.integers(0, 1024, 3000).astype(np.uint32)
    p1, s1 = model.encode(ids, n_segments=4)
    p2, s2 = model.encode(ids, n_segments=4, max_batch_tokens=600)
    assert p1 == p2 and np.array_equal(s1, s2)
    for g in range(4):
        solo, _ = model.encode(ids[int(s1[g]) : int(s1[g + 1])], n_segments=1)
        assert solo[0] == p1[g]


def test_tiny_xe_bits_vs_oracle(gpu_ctx):
    model = _tiny(gpu_ctx, _lib.CZ_ENGINE_TCGEN05, embed_std=0.2)
    rng = np.random.default_rng(6)
    hist = rng.integers(0, 1024, 600).astype(np.uint32)
    targets = rng.integers(0, 1024, 64).astype(np.uint32)
    hint = rng.integers(0, 1024, 127).astype(np.uint32)
    jobs = [(cz.xe_make_prime(hist, None), targets), (cz.xe_make_prime(hist, hint), targets), (cz.xe_make_prime(hist[:5], hint[:3]), targets[:7])]
    got = model.xe_bits(jobs)
    orc = _oracle_for(model, round_bf16=1)
    want = [orc.xe_bits(hist, targets), orc.xe_bits(hist, targets, hint), orc.xe_bits(hist[:5], targets[:7], hint[:3])]
    for a, b in zip(got, want):
        assert abs(a - b) <= 0.01 * b, (a, b)


def test_full_size_smollm_parity_and_roundtrip(gpu_ctx):
    """SmolLM-135M shape (random-init): logits vs the oracle on a few positions, then a 2-segment round trip."""
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.05)
    rng = np.random.default_rng(0)
    prime = rng.integers(0, 49152, 6).astype(np.uint32)
    targets = rng.integers(0, 49152, 3).astype(np.uint32)
    got = model.chunk_logits(prime, targets)
    orc = _oracle_for(model, round_bf16=1)
    want = [orc.reprime(prime)] + [orc.step_logits(t) for t in targets[:-1]]
    for j in range(3):
        assert np.abs(got[j] - want[j]).max() < 0.03 * max(1.0, np.abs(want[j]).max()), j
    ids = rng.integers(0, 49152, 1200).astype(np.uint32)
    pays, seg_start = model.encode(ids, n_segments=2)
    out = model.decode(pays, seg_start)
    assert np.array_equal(out, ids)


# ------------------------------------------------------------------ RWKV-7 (SURVEY 8 a-5)
def _rwkv_tiny(gpu_ctx, engine=_lib.CZ_ENGINE_TCGEN05, seed=7):
    import sys

    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from rwkv7_weights import RWKV7_TINY, make_weights

    W = make_weights(RWKV7_TINY, seed)
    model = cz.Model(gpu_ctx, RWKV7_TINY, engine=engine)
    for name, arr in W.items():
        model.set_tensor(name, arr)
    return model, RWKV7_TINY, W


@pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])
def test_rwkv7_tiny_logits_vs_oracle_and_golden(gpu_ctx, engine):
    """CUDA RWKV-7 (bf16 GEMM operands, fp32 state / accumulate) vs the f32 oracle, the oracle with the same bf16 rounding
    points, and the fla-composed golden.  Stated tolerance: max|delta| <= 0.05 * std(logits) vs f32, 0.03 * std vs bf16-rounded."""
    model, cfg, W = _rwkv_tiny(gpu_ctx, engine)
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rwkv7_tiny_golden.npz"))
    toks = z["tokens"].astype(np.uint32)
    got = model.chunk_logits(toks[:1], toks[1:])  # column j = logits after toks[0..j]
    o32 = oracle.Session.rwkv7(cfg, W, round_bf16=0)
    o16 = oracle.Session.rwkv7(cfg, W, round_bf16=1)
    for j in range(len(toks) - 1):
        w32, w16 = o32.step_logits(toks[j]), o16.step_logits(toks[j])
        sd = z["logits"][j].std()
        assert np.abs(got[j] - w16).max() < 0.03 * sd, (j, np.abs(got[j] - w16).max() / sd)
        assert np.abs(got[j] - w32).max() < 0.05 * sd, j
        assert np.abs(got[j] - z["logits"][j]).max() < 0.05 * sd, j


@pytest.mark.parametrize("engine,n", [(_lib.CZ_ENGINE_SIMT, 90), (_lib.CZ_ENGINE_TCGEN05, 90), (_lib.CZ_ENGINE_TCGEN05, 2048)],
                         ids=["simt", "tc", "tc-long"])
def test_rwkv7_stepwise_equals_slab_bitwise(gpu_ctx, engine, n):
    """decode safety: T=1 steps, one long slab and several short slabs give bit-identical logits (the long case carries the
    recurrent state over 2,047 steps)"""
    model, cfg, _ = _rwkv_tiny(gpu_ctx, engine)
    rng = np.random.default_rng(21)
    toks = rng.integers(0, cfg["vocab"], n).astype(np.uint32)
    slab = model.chunk_logits(toks[:1], toks[1:])
    s = model.session()
    step = np.stack([s.step_logits_tensor(t) for t in toks[:-1]])
    assert np.array_equal(slab.view(np.uint32), step.view(np.uint32))
    assert s.index_pos() == len(toks) - 1
    # reprime = fresh state + replay (src/models.rs:162-170)
    again = s.reprime_with_history_and_get_last_logits_tensor(toks[:40])
    assert np.array_equal(again.view(np.uint32), slab[39].view(np.uint32))
    assert s.index_pos() == 40


@pytest.mark.parametrize("n,n_seg,lit", [(1, 1, 0.0), (400, 1, 0.0), (900, 3, 0.08), (257, 5, 0.3), (4096, 4, 0.05)])
def test_rwkv7_roundtrip_and_oracle_bitstream(gpu_ctx, n, n_seg, lit):
    model, cfg, W = _rwkv_tiny(gpu_ctx)
    V = cfg["vocab"]
    rng = np.random.default_rng(n + n_seg)
    ids = rng.integers(0, V, n).astype(np.uint32)
    mask = rng.random(n) < lit
    ids[mask] = V + rng.integers(0, 256, int(mask.sum()))  # literal-escape symbols (src/main.rs:833-895)
    pays, seg_start = model.encode(ids, n_segments=n_seg)
    # (1) GPU logits -> ORACLE literal-mode quantiser + ORACLE coder == GPU payload of segment 0
    a, b = int(seg_start[0]), int(seg_start[1])
    logits = model.chunk_logits([0], ids[a:b])
    bounds = [tuple(int(x) for x in oracle.logits_to_cdf(logits[j], 1)[[ids[a + j], ids[a + j] + 1]]) for j in range(b - a)]
    assert oracle.ac_encode(bounds) == pays[0]
    # (2) slab-shape invariance: a small row budget forces many time slabs
    pays2, _ = model.encode(ids, n_segments=n_seg, max_batch_tokens=max(n_seg * 7, 16))
    assert pays2 == pays
    # (3) round trip through the lock-step decoder (literals do not step the model)
    out = model.decode(pays, seg_start)
    assert np.array_equal(out, ids)
    # (4) compressed size vs the f32 CPU oracle running the reference loop
    if n >= 400 and n_seg == 1:
        orc = oracle.Session.rwkv7(cfg, W)
        ref_payload, _ = orc.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32), backend=1)
        assert abs(len(pays[0]) - len(ref_payload)) <= 0.005 * len(ref_payload) + 2


def test_rwkv7_xe_bits_vs_oracle(gpu_ctx):
    model, cfg, W = _rwkv_tiny(gpu_ctx)
    V = cfg["vocab"]
    rng = np.random.default_rng(16)
    hist = rng.integers(0, V, 200).astype(np.uint32)
    hist[rng.random(200) < 0.05] = V + 7  # literals are filtered out of the history (src/main.rs:1763-1765)
    targets = rng.integers(0, V, 48).astype(np.uint32)
    targets[5] = V + 65
    hint = rng.integers(0, V, 30).astype(np.uint32)
    big = 1 << 30  # max_context_length() == usize::MAX for RWKV (src/models.rs:150): the whole history is the prime
    jobs = [(cz.xe_make_prime(hist, None, big), targets), (cz.xe_make_prime(hist, hint, big), targets)]
    got = model.xe_bits(jobs)
    orc = oracle.Session.rwkv7(cfg, W, round_bf16=1)
    want = [orc.xe_bits(hist, targets, None, backend=1), orc.xe_bits(hist, targets, hint, backend=1)]
    for g, w in zip(got, want):
        assert abs(g - w) <= 0.01 * w, (g, w)


def test_rwkv7_hint_prime_event_matches_oracle_loop(gpu_ctx):
    """a gated hint prime resets the state and re-feeds the prime (src/main.rs:2137-2149): payload == oracle loop on GPU logits
    is covered above; here the event path must equal encoding the two halves as independent units"""
    model, cfg, W = _rwkv_tiny(gpu_ctx)
    rng = np.random.default_rng(31)
    ids = rng.integers(0, cfg["vocab"], 300).astype(np.uint32)
    prime = rng.integers(0, cfg["vocab"], 20).astype(np.uint32)
    pays, _ = model.encode(ids, n_segments=1, events=[(120, prime, 120 + 64)])
    orc = oracle.Session.rwkv7(cfg, W)
    ref, _ = orc.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32), backend=1, events=[(120, prime, 184)])
    assert abs(len(pays[0]) - len(ref)) <= 0.005 * len(ref) + 2
    # bit-exact against the oracle coder fed with the GPU's own logits
    l1 = model.chunk_logits([0], ids[:120])
    l2 = model.chunk_logits(prime, ids[120:])
    logits = np.concatenate([l1, l2])
    bounds = [tuple(int(x) for x in oracle.logits_to_cdf(logits[j], 1)[[ids[j], ids[j] + 1]]) for j in range(300)]
    assert oracle.ac_encode(bounds) == pays[0]


def test_hint_prime_events_roundtrip_both_backends(gpu_ctx):
    """SURVEY 8 a-7: gated hint primes in the main stream (src/main.rs:2123-2149 encode, 2586-2614 decode): the prime replaces
    the context, `hold_until` suppresses the next context re-prime; the batched decoder must follow the same schedule."""
    rng = np.random.default_rng(41)
    # SmolLM: events at a chunk-interior index and right before a re-prime boundary that the hold-off then suppresses
    model = _tiny(gpu_ctx, _lib.CZ_ENGINE_TCGEN05)
    ids = rng.integers(0, 1024, 1500).astype(np.uint32)
    ev = [(200, rng.integers(0, 1024, 300).astype(np.uint32), 200 + 512), (900, rng.integers(0, 1024, 63).astype(np.uint32), 900 + 512)]
    pays, seg = model.encode(ids, n_segments=1, events=ev)
    plain, _ = model.encode(ids, n_segments=1)
    assert pays != plain
    orc = _oracle_for(model, round_bf16=0)
    ref, rep = orc.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32), events=ev)
    assert abs(len(pays[0]) - len(ref)) <= 0.005 * len(ref) + 2
    assert np.array_equal(model.decode(pays, seg, events=ev), ids)
    # RWKV-7: a prime resets the recurrent state (src/models.rs:162-170)
    rmodel, cfg, _ = _rwkv_tiny(gpu_ctx)
    rid = rng.integers(0, cfg["vocab"], 400).astype(np.uint32)
    rev = [(0, rng.integers(0, cfg["vocab"], 9).astype(np.uint32), 64), (150, rng.integers(0, cfg["vocab"], 40).astype(np.uint32), 214)]
    rp, rs = rmodel.encode(rid, n_segments=1, events=rev)
    assert np.array_equal(rmodel.decode(rp, rs, events=rev), rid)


def test_gate_scan_paired_streams_vs_oracle_and_roundtrip(gpu_ctx):
    """BASELINE config 4 in miniature: the agentic gate replayed from cached agent texts.  All baseline / hint-conditioned
    cross-entropy evaluations of all boundaries run as ONE batch of paired streams (src/main.rs:2043-2054), the gated
    boundaries become hint primes of the main stream (2123-2149), the container carries AGT2 records, and the decoder
    rebuilds the same primes from the records + what it has decoded (2586-2614)."""
    from candlezip_b200 import container, gate

    model = _tiny(gpu_ctx, _lib.CZ_ENGINE_TCGEN05)  # flat-ish logits: random tokens must not hit zero-width intervals
    rng = np.random.default_rng(77)
    ids = rng.integers(0, 1024, 1400).astype(np.uint32)
    # "agent texts": strings whose characters map to token ids (a stand-in for tokenizer + agent, both absent offline)
    tok = lambda s, m: [(ord(ch) * 7) % 1024 for ch in s][:m]
    texts = {1: "Alpha Beta 12 gamma " * 9, 2: "", 3: "Delta 7 Epsilon " * 30, 5: "Zeta"}
    pays, seg, records, rows, events = gate.scan_encode(model, ids, texts, tok, agent_chunk=256, scan_lookahead=200)
    assert len(records) == 5 and [r["chunk_index"] for r in rows] == [1, 2, 3, 4, 5]
    # (1) XE parity of the paired streams against the oracle running cross_entropy_bits_over_span
    orc = _oracle_for(model, round_bf16=1)
    seq = np.concatenate([[0], ids]).astype(np.uint32)
    jobs, plan = gate.plan_scan(ids, texts, tok, 256, 200)
    bits = model.xe_bits(jobs)
    for e in plan[:3]:
        i = e["i"]
        hist, targets = seq[max(0, i - 511):i], seq[i:min(i + 200, len(seq))]
        want = orc.xe_bits(hist, targets)
        assert abs(bits[e["job0"]] - want) <= 0.01 * want
        slot = e["slots"][0 * 4 + 1]
        if slot is not None:
            want_c = orc.xe_bits(hist, targets, e["hints"][0][:127])
            assert abs(bits[slot] - want_c) <= 0.01 * want_c
    assert rows[1]["gate"] == 0 and rows[1]["bits_saved"] == 0.0 and rows[3]["gate"] == 0   # empty hints never gate
    # (2) the gated stream decodes in one call from (records, agent texts) alone
    hints = [e["hints"] for e in plan]
    dec_events = gate.events_from_records(records, hints, 256, len(ids), scan_lookahead=200)
    assert len(dec_events) == len(events) == sum(r & 1 for r in records)
    assert np.array_equal(model.decode(pays, seg, events=dec_events or None), ids)
    # (3) the same schedule on the oracle (explicit primes) gives the same compressed size within 0.5 %
    ev_explicit = [(i, np.concatenate([seq[i + 1 - ht:i + 1], h]).astype(np.uint32), hold) for (i, h, hold, ht) in events]
    ref, _ = _oracle_for(model, round_bf16=0).encode_tokens(seq, events=ev_explicit)
    assert abs(len(pays[0]) - len(ref)) <= 0.005 * len(ref) + 2
    # (4) container with the AGT2 section (flag bit 2), byte layout of src/main.rs:658-670
    blob = container.write_container(dict(token_count=len(ids), orig_len_bytes=len(ids), vocab_size=1024, reserved_flags=1), b"m", pays,
                                     gates=records)
    f, _, g, _, _, p2 = container.read_container(blob)
    assert g == records and p2 == pays and f["reserved_flags"] & 4


def test_file_level_compress_decompress_both_backends(gpu_ctx):
    """bytes -> container -> bytes (the reference's compress / decompress / self-test, src/main.rs:156-221, minus the CLI):
    byte-level SmolLM (every input round-trips, incl. non-UTF-8), RWKV-7 with a trie vocabulary + literal escapes, segmented
    containers, header fields, and the BLAKE3 check of the decoded bytes that the reference never performs."""
    from candlezip_b200 import codec, container

    rng = np.random.default_rng(9)
    text = (b"It was the best of times, it was the worst of times. " * 40) + bytes(rng.integers(0, 256, 300, dtype=np.uint8))
    model = _tiny(gpu_ctx, _lib.CZ_ENGINE_TCGEN05)
    for nseg in (1, 4):
        blob = codec.compress(model, text, n_segments=nseg)
        f, rep, gates, eng, st, pays = container.read_container(blob)
        assert f["token_count"] == len(text) and f["orig_len_bytes"] == len(text) and f["vocab_size"] == 1024
        assert f["context_window"] == 512 and f["reprime_interval"] == 512 and f["orig_hash16"] == container.blake3_16(text)
        assert (st is None) == (nseg == 1) and len(pays) == nseg
        assert codec.decompress(model, blob) == text
    bad = bytearray(blob)
    bad[-3] ^= 0x10  # corrupt the payload: decode yields other bytes, caught by the hash check
    with pytest.raises((ValueError, cz.CzError)):
        codec.decompress(model, bytes(bad))
    assert codec.decompress(model, codec.compress(model, b"")) == b""
    # RWKV-7 with a toy trie vocabulary (ids < 320) and bytes the vocabulary cannot express
    import test_cpu_oracle as tco

    rmodel, cfg, _ = _rwkv_tiny(gpu_ctx)
    tok = codec.RwkvTokenizer(tco._toy_rwkv_vocab())
    rtext = b"the thing in the abcd " * 30
    rblob = codec.compress(rmodel, rtext, tokenizer=tok, n_segments=2)
    assert codec.decompress(rmodel, rblob, tokenizer=tok) == rtext
    assert container.read_container(rblob)[0]["token_count"] < len(rtext)  # multi-byte tokens
    gap = b"abc\xffdef the end"
    gblob = codec.compress(rmodel, gap, tokenizer=tok)
    assert container.read_container(gblob)[0]["token_count"] == len(gap)  # every byte a literal escape
    assert codec.decompress(rmodel, gblob, tokenizer=tok) == gap


def test_full_size_smollm_multi_chunk_invariance_and_roundtrip(gpu_ctx):
    """BASELINE config 2 shape in miniature at FULL model size: many segments, several reprime chunks each.  Size-independent
    properties: identical bytes whatever the wave size; a segment's stream equals the single-stream encode of its tokens
    (batch-size invariance); decode(encode(x)) == x through the lock-step decoder (graph-replayed steps, chunk re-primes)."""
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    rng = np.random.default_rng(5)
    n, nseg = 24 * 1100, 24
    ids = rng.integers(0, 256, n).astype(np.uint32)  # byte-level ids, like the bench
    p1, s1 = model.encode(ids, n_segments=nseg)
    p2, s2 = model.encode(ids, n_segments=nseg, max_batch_tokens=9000)
    assert p1 == p2 and np.array_equal(s1, s2)
    solo, _ = model.encode(ids[int(s1[3]) : int(s1[4])], n_segments=1)
    assert solo[0] == p1[3]
    assert np.array_equal(model.decode(p1, s1), ids)
    # long reprime interval: one chunk of 511 + 3000 positions (beyond the old 2000-position limit of the mma.sync kernel)
    long_ids = rng.integers(0, 256, 3600).astype(np.uint32)
    pl, sl = model.encode(long_ids, n_segments=1, reprime_interval=3000)
    assert np.array_equal(model.decode(pl, sl, reprime_interval=3000), long_ids)


def test_cli_twin_self_test(gpu_ctx, tmp_path):
    """`python -m candlezip_b200 self-test` (src/main.rs:156-221) on a small file, both backends, segmented"""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = tmp_path / "sample.txt"
    p.write_bytes((b"the quick brown fox jumps over the lazy dog. " * 30) + bytes(range(256)))
    for backend in ("smollm", "rwkv7"):
        r = subprocess.run([sys.executable, "-m", "candlezip_b200", "self-test", str(p), "--backend", backend, "--segments", "4"], cwd=root,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "roundtrip OK" in r.stdout, (r.stdout, r.stderr[-500:])


def test_rwkv7_full_size_roundtrip(gpu_ctx):
    """rwkv7-g1-0.1b shape (random-init): logits vs the oracle on a few positions, then a multi-segment round trip."""
    model = cz.Model(gpu_ctx, cz.RWKV7_0P1B).random_init(3, 0.02, 0.05)
    cfg = dict(cz.RWKV7_0P1B)
    rng = np.random.default_rng(0)
    toks = rng.integers(0, 65536, 6).astype(np.uint32)
    got = model.chunk_logits(toks[:1], toks[1:])
    orc = oracle.Session.rwkv7(cfg, model.tensors(), round_bf16=1)
    for j in range(5):
        want = orc.step_logits(toks[j])
        assert np.abs(got[j] - want).max() < 0.03 * max(1.0, np.abs(want).max()), j
    ids = rng.integers(0, 65536, 1500).astype(np.uint32)
    pays, seg_start = model.encode(ids, n_segments=3)
    out = model.decode(pays, seg_start)
    assert np.array_equal(out, ids)
