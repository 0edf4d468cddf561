"""Deep RWKV-7 parity (-m gpu): the WKV-7 scan and LayerNorm-mix kernels alone against an f64 restatement (tests/rwkv7_ref.py) at
the shapes, decays and rows where they could go wrong, their stream / slot / split structure bit for bit, every position of long
BOS-started runs against the oracle, and bits per token on text drawn from the model itself.

RWKV-7 carries one recurrent state through a whole segment and never reprimes, so an error that builds up along the run, or that
only the 8-element-per-lane LayerNorm-mix (d_model a multiple of 256, the 0.1B model's 768) makes, is invisible to short tests.
The tolerances are 2x maxima measured on a B200 by scripts/rwkv_parity_report.py (profiles/rwkv_parity_r09.md)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
import parity_util as pu
import rwkv7_ref as rr
from candlezip_b200 import _lib

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from rwkv7_weights import RWKV7_TINY, bf16_exact, long_memory, make_weights  # noqa: E402

pytestmark = pytest.mark.gpu

# ---- tolerances measured on a B200 (profiles/rwkv_parity_r09.md); each is 2x the named row's maximum unless said otherwise
TOL_SCAN_ROW = 2 * 2.6e-6          # "scan vs f64, max over rows": error beyond the bf16 rounding of the output / std(ref row)
TOL_SCAN_STATE = 2 * 1.05e-6       # "final state": max|dS| / max|S| over the six SCAN_SHAPES
# model level, max|logit - oracle| / std(oracle logits) per position, split into the first 512-position block (a run starts
# from a zero state, where the bf16 rounding points move the 0.1B logits most: the oracle against itself reaches 0.59 there)
# and the positions after it: ((bf16 oracle: first block, after), (f32 oracle: first block, after)), max over engines
TOLS = {
    "RWKV7_TINY seed 7": ((2 * 0.0236, 2 * 0.0252), (2 * 0.0384, 2 * 0.0503)),
    "long memory": ((2 * 0.0223, 2 * 0.0288), (2 * 0.0404, 2 * 0.0371)),
    "d_model 256": ((2 * 0.0201, 2 * 0.0311), (2 * 0.1279, 2 * 0.0423)),
    "0.1B shape": ((2 * 0.2616, 2 * 0.0718), (2 * 0.7339, 2 * 0.0889)),
}

u16p = C.POINTER(C.c_uint16)
i32p = C.POINTER(C.c_int)
f32p = C.POINTER(C.c_float)
ROW_NAMES = ("r", "k", "v", "wl", "al", "vl", "g")
VEC_NAMES = ("w0", "a0", "v0", "k_k", "k_a", "r_k", "gn_w", "gn_b")
BF16_SENTINEL = 0x7FA5  # a NaN pattern no kernel writes
F32_SENTINEL = np.uint32(0x7FC0BEEF)


def _i32(a):
    return np.ascontiguousarray(a, np.int32)


# ------------------------------------------------------------------------------------------------------------ WKV-7 scan hook
def run_scan(ctx, layer0, rows, vf, vecs, state, row_begin, row_end, stream_slot, active=None, out=None):
    """One cz_test_wkv7_scan call.  rows [7][R][C], vf [R][C], vecs [8][C], state [n_slots][H][4096] (kernel layout), all f32.
    Returns (out bf16 bits [R][C], v_first, state) -- fresh arrays; out starts as `out` (default: the sentinel)."""
    rows = np.ascontiguousarray(rows, np.float32)
    R, Cw = rows.shape[1], rows.shape[2]
    H = Cw // 64
    vf = np.array(vf, np.float32)
    st = np.array(state, np.float32)
    o = np.full((R, Cw), BF16_SENTINEL, np.uint16) if out is None else np.array(out, np.uint16)
    rb, re, sl = _i32(row_begin), _i32(row_end), _i32(stream_slot)
    act = None if active is None else _i32(active)
    _lib.check(_lib.lib.cz_test_wkv7_scan(
        ctx._h, int(layer0), R, H, len(rb), rb.ctypes.data_as(i32p), re.ctypes.data_as(i32p), sl.ctypes.data_as(i32p),
        None if act is None else act.ctypes.data_as(i32p), st.shape[0], rows.ctypes.data_as(f32p), vf.ctypes.data_as(f32p),
        np.ascontiguousarray(vecs, np.float32).ctypes.data_as(f32p), st.ctypes.data_as(f32p), o.ctypes.data_as(u16p)))
    return o, vf, st


def scan_case(rng, T, H):
    """Row inputs of T rows with every class of row the scan must survive, in blocks of T/16 rows cycling through the classes:
    plain; long memory (z = wl + w0 in [-14, -9]: 1 - w < 1e-4); z < -88.7 (exp(-z) overflows, w == 1); z >> 0 (w -> e^-e^-0.5);
    a near 0; a near 1; k . k_k tiny (nrm ~1e-5, far below 1 but above the 1e-12 floor) or zero in one head, r == 0 rows; g == 0
    rows; small r (the head's outputs have a variance near the group-norm eps)."""
    Cw = 64 * H
    vecs = np.stack([rng.normal(-1.0, 1.5, Cw), rng.normal(0, 1, Cw), rng.normal(0, 1, Cw), rng.normal(0.85, 0.1, Cw),
                     rng.normal(1.0, 0.1, Cw), rng.normal(0, 0.3, Cw), rng.normal(1.0, 0.1, Cw), rng.normal(0, 0.1, Cw)]).astype(np.float32)
    rows = rng.normal(0, 1, (7, T, Cw)).astype(np.float32)
    r, k, v, wl, al, vl, g = rows
    w0 = vecs[0]
    blk = max(1, T // 16)
    for t0 in range(0, T, blk):
        s = slice(t0, min(T, t0 + blk))
        cls = (t0 // blk) % 9
        n = s.stop - s.start
        if cls == 1:
            wl[s] = rng.uniform(-14, -9, (n, Cw)) - w0
        elif cls == 2:
            wl[s] = -100.0 - np.abs(w0)
        elif cls == 3:
            wl[s] = 40.0 + np.abs(w0)
        elif cls == 4:
            al[s] = -40.0
        elif cls == 5:
            al[s] = 40.0
        elif cls == 6:
            k[s, :64] *= 1e-6
            k[s.start + 1:s.stop:3, 64 * (H - 1):] = 0.0
            r[s.start + 2:s.stop:5] = 0.0
        elif cls == 7:
            g[s.start::2][: (n + 1) // 2] = 0.0
        elif cls == 8:
            r[s] *= np.where(np.arange(n) % 2 == 0, 1e-3, 3e-4)[:, None].astype(np.float32)
    return rows, vecs


def _vecs_dict(vecs):
    return {n: vecs[i].astype(np.float64) for i, n in enumerate(VEC_NAMES)}


def scan_ref(rows, vf, vecs, state, layer0):
    """f64 reference of one stream over all rows: returns (out [T][C], v_first [T][C], state [H][64][64])"""
    S = rr.state_from_kernel(np.asarray(state, np.float64))
    rd = {n: rows[i].astype(np.float64) for i, n in enumerate(ROW_NAMES)}
    out, vfo = rr.wkv7_scan(S, rd, np.asarray(vf, np.float64), _vecs_dict(vecs), layer0)
    return out, vfo, S


def scan_metrics(out16, ref_out, st, ref_S):
    """(per row: max over the row of the error beyond the bf16 rounding of the output, (|out - ref| - ulp_bf16(ref) / 2)+ / std(ref
    row), over rows whose reference is not identically zero; final state max|dS| / max|S|)"""
    got = pu.bf16_to_f32(out16).astype(np.float64)
    sd = ref_out.std(axis=1)
    live = sd > 0
    row = np.maximum(np.abs(got - ref_out) - 0.5 * bf16_ulp(ref_out), 0.0).max(axis=1)[live] / sd[live]
    S = rr.state_from_kernel(st.astype(np.float64))
    return row, np.abs(S - ref_S).max() / np.abs(ref_S).max()


SCAN_SHAPES = [(2, True, False), (2, False, True), (12, True, True), (12, False, False), (16, True, False), (16, False, True)]


def scan_vs_f64(ctx, H, layer0, nonzero_init, T=4096, seed=0):
    rng = np.random.default_rng(seed * 97 + H * 2 + int(layer0) + 4 * int(nonzero_init))
    rows, vecs = scan_case(rng, T, H)
    vf = rng.normal(0, 1, (T, 64 * H)).astype(np.float32)
    S0 = rr.state_to_kernel(rng.normal(0, 0.5, (1, H, 64, 64)) if nonzero_init else np.zeros((1, H, 64, 64))).astype(np.float32)
    out, vfo, st = run_scan(ctx, layer0, rows, vf, vecs, S0, [0], [T], [0])
    ref_out, ref_vf, ref_S = scan_ref(rows, vf, vecs, S0[0], layer0)
    row, smet = scan_metrics(out, ref_out, st[0], ref_S)
    return dict(rows=rows, vf_in=vf, out=out, vf=vfo, ref_out=ref_out, row=row, state=smet)


@pytest.mark.parametrize("H,layer0,nonzero_init", SCAN_SHAPES)
def test_rwkv7_deep_scan_vs_f64(gpu_ctx, H, layer0, nonzero_init):
    """4,096 rows of one stream through every class of scan_case, per row and for the final state"""
    r = scan_vs_f64(gpu_ctx, H, layer0, nonzero_init)
    assert np.all(np.isfinite(pu.bf16_to_f32(r["out"])))
    g = r["rows"][6]
    assert np.all(r["out"][g == 0] & 0x7FFF == 0), "a zero gate must give a zero output"
    assert r["row"].max() < TOL_SCAN_ROW, (int(r["row"].argmax()), float(r["row"].max()))
    assert r["state"] < TOL_SCAN_STATE, r["state"]
    if layer0:
        assert np.array_equal(r["vf"].view(np.uint32), r["rows"][2].view(np.uint32)), "layer 0 must hand v over as v_first bit for bit"
    else:
        assert np.array_equal(r["vf"].view(np.uint32), r["vf_in"].view(np.uint32)), "layers > 0 only read v_first"


def test_rwkv7_deep_scan_decay_edges_exact(gpu_ctx):
    """one row with k == 0 (so the state only decays: S' = S * w) from a non-zero state: z < -88.7 must keep the state bit for bit
    (w == 1 exactly); z = -12 scales it by 1 - 3.7e-6; z >> 0 by e^-e^-0.5"""
    H = 2
    rng = np.random.default_rng(5)
    S0 = rr.state_to_kernel(rng.normal(0, 1, (1, H, 64, 64))).astype(np.float32)
    for z, want in ((-100.0, 1.0), (-12.0, rr.decay(np.array([-12.0]))[0]), (40.0, np.exp(-np.exp(-0.5)))):
        rows, vecs = scan_case(np.random.default_rng(6), 1, H)
        rows[1] = 0.0
        vecs[0] = 0.0
        rows[3] = z
        _, _, st = run_scan(gpu_ctx, False, rows, np.zeros((1, 64 * H)), vecs, S0, [0], [1], [0])
        if want == 1.0:
            assert np.array_equal(st.view(np.uint32), S0.view(np.uint32)), "w must be exactly 1 where exp(-z) overflows"
        else:
            ratio = st.astype(np.float64)[S0 != 0] / S0.astype(np.float64)[S0 != 0]
            assert np.abs(ratio - want).max() < 2e-7, (z, float(np.abs(ratio - want).max()))


def _stream_layout(lengths):
    ends = np.cumsum(lengths)
    return ends - np.asarray(lengths), ends, int(ends[-1])


def test_rwkv7_deep_scan_streams_slots_and_independence(gpu_ctx):
    """7 streams of lengths {0, 1, 2, 31, 32, 33, 500} in one launch, slots permuted into 9 slots, one stream inactive: every
    active stream equals that stream run alone (bitwise: output, v_first and state); unused and inactive slots, the inactive
    stream's output rows and the rows of the empty stream keep their sentinels"""
    H = 2
    rng = np.random.default_rng(8)
    lengths = [31, 0, 500, 1, 33, 2, 32]
    rb, re, R = _stream_layout(lengths)
    slot = np.array([4, 0, 7, 2, 8, 5, 1])
    active = np.array([1, 1, 1, 1, 0, 1, 1])  # the 33-row stream does not step
    rows, vecs = scan_case(rng, R, H)
    vf = rng.normal(0, 1, (R, 64 * H)).astype(np.float32)
    S0 = rng.normal(0, 0.5, (9, H, 4096)).astype(np.float32)
    S0[[3, 6]].view(np.uint32)[:] = F32_SENTINEL
    for layer0 in (True, False):
        out, vfo, st = run_scan(gpu_ctx, layer0, rows, vf, vecs, S0, rb, re, slot, active)
        for u in (3, 6, slot[4], slot[1]):  # unused, inactive, empty
            assert np.array_equal(st[u].view(np.uint32), S0[u].view(np.uint32)), u
        assert np.all(out[rb[4]:re[4]] == BF16_SENTINEL)
        assert np.array_equal(vfo[rb[4]:re[4]].view(np.uint32), vf[rb[4]:re[4]].view(np.uint32))
        for s in range(7):
            if not active[s] or lengths[s] == 0:
                continue
            a, b = rb[s], re[s]
            o1, vf1, st1 = run_scan(gpu_ctx, layer0, rows[:, a:b], vf[a:b], vecs, S0[slot[s]][None], [0], [b - a], [0])
            assert np.array_equal(out[a:b], o1), (layer0, s)
            assert np.array_equal(vfo[a:b].view(np.uint32), vf1.view(np.uint32)), (layer0, s)
            assert np.array_equal(st[slot[s]].view(np.uint32), st1[0].view(np.uint32)), (layer0, s)
        # other neighbours (disjoint rows, other slots) change nothing for stream 2
        out2, _, st2 = run_scan(gpu_ctx, layer0, rows, vf, vecs, S0[[7, 0, 5]], [rb[2], 0, re[2]], [re[2], 31, R], [0, 1, 2])
        assert np.array_equal(out2[rb[2]:re[2]], out[rb[2]:re[2]]) and np.array_equal(st2[0].view(np.uint32), st[7].view(np.uint32))


@pytest.mark.parametrize("H,layer0", [(2, True), (12, False)])
def test_rwkv7_deep_scan_splits_bitwise(gpu_ctx, H, layer0):
    """decode safety at kernel level: T rows in one launch == the same rows over several launches with the state carried ==
    T single-row launches, bit for bit"""
    T = 160
    rng = np.random.default_rng(10 + H)
    rows, vecs = scan_case(rng, T, H)
    vf = rng.normal(0, 1, (T, 64 * H)).astype(np.float32)
    S0 = rng.normal(0, 0.5, (1, H, 4096)).astype(np.float32)
    whole, vfw, stw = run_scan(gpu_ctx, layer0, rows, vf, vecs, S0, [0], [T], [0])
    for cuts in ([0, 37, 101, T], list(range(T + 1))):
        st = S0
        parts, vfs = [], []
        for a, b in zip(cuts[:-1], cuts[1:]):
            o, v1, st = run_scan(gpu_ctx, layer0, rows[:, a:b], vf[a:b], vecs, st, [0], [b - a], [0])
            parts.append(o)
            vfs.append(v1)
        assert np.array_equal(np.concatenate(parts), whole), len(cuts)
        assert np.array_equal(np.concatenate(vfs).view(np.uint32), vfw.view(np.uint32))
        assert np.array_equal(st.view(np.uint32), stw.view(np.uint32)), len(cuts)


# ------------------------------------------------------------------------------------------------------------ LayerNorm-mix hook
def run_ln_mix(ctx, nmix, form, in_place, x, lnw, lnb, mu, prev_row, slot, flags, state_in, state_out, eps=1e-5):
    x = np.ascontiguousarray(x, np.float32)
    R, Cw = x.shape
    si = np.ascontiguousarray(state_in, np.float32)
    so = np.array(state_out, np.float32)
    out = np.empty((nmix, R, Cw), np.uint16)
    used = C.c_int(-1)
    pr, sl, fl = _i32(prev_row), _i32(slot), _i32(flags)
    _lib.check(_lib.lib.cz_test_rwkv_ln_mix(
        ctx._h, nmix, form, int(in_place), R, Cw, si.shape[0], x.ctypes.data_as(f32p), np.ascontiguousarray(lnw, np.float32).ctypes.data_as(f32p),
        np.ascontiguousarray(lnb, np.float32).ctypes.data_as(f32p), np.ascontiguousarray(mu, np.float32).ctypes.data_as(f32p),
        pr.ctypes.data_as(i32p), sl.ctypes.data_as(i32p), fl.ctypes.data_as(i32p), si.ctypes.data_as(f32p), so.ctypes.data_as(f32p),
        C.c_float(eps), out.ctypes.data_as(u16p), C.byref(used)))
    return out, so, used.value


def ln_mix_case(rng, Cw, nmix, in_place):
    """Rows in chains through prev_row (a chain's first row reads state_in[slot]); the last row of a chain writes state_out[slot]
    (flags bit 0) unless bit 1 suppresses it; three edge rows: a constant row (variance 0), one outlier at 1e3 x and a row offset by
    100 sigma.  in_place: every row is its own chain with its own slot, as in the stepwise decoder."""
    if in_place:
        R = 32
        chains = [[r] for r in range(R)]
        flags = np.where(np.arange(R) % 4 == 3, 3, 1)
    else:
        chains = [list(range(0, 9)), [9], list(range(10, 21)), list(range(21, 30)), [30, 31], list(range(32, 40))]
        R = 40
        flags = np.zeros(R, np.int32)
        for c, f in zip(chains, (1, 1, 3, 1, 0, 1)):
            flags[c[-1]] = f
    prev = np.full(R, -1)
    slot = np.zeros(R, np.int32)
    n_slots = R if in_place else 8
    chain_slot = np.arange(R) if in_place else [3, 0, 5, 6, 1, 7]
    for c, s in zip(chains, chain_slot):
        for j, r in enumerate(c):
            slot[r] = s
            prev[r] = c[j - 1] if j else -1
    x = rng.normal(0, 1, (R, Cw)).astype(np.float32)
    edge = np.array([8, 13, 29])  # 8 and 29 end a chain (their LayerNorm is written), 13 is the previous token of 14
    x[8] = np.float32(0.1)
    x[13, 17] = 1e3
    x[29] += 100.0
    lnw = rng.normal(1.0, 0.1, Cw).astype(np.float32)
    lnb = rng.normal(0.0, 0.1, Cw).astype(np.float32)
    mu = rng.uniform(0, 1, (nmix, Cw)).astype(np.float32)
    state_in = rng.normal(0, 1, (n_slots, Cw)).astype(np.float32)
    return x, lnw, lnb, mu, prev, slot, flags, state_in, edge


def ln_mix_ref(x, lnw, lnb, mu, prev, slot, state_in, eps=1e-5):
    xn = rr.layer_norm(x.astype(np.float64), lnw.astype(np.float64), lnb.astype(np.float64), eps)
    pv = np.where((prev >= 0)[:, None], xn[np.maximum(prev, 0)], state_in[slot].astype(np.float64))
    return xn, pv, np.stack([rr.token_shift_mix(xn, pv, m.astype(np.float64)) for m in mu])


def bf16_ulp(a):
    a = np.abs(np.asarray(a, np.float64))
    return np.exp2(np.floor(np.log2(np.maximum(a, 2.0 ** -126))) - 7)


def ln_mix_metrics(out, so, xn_ref, pv_ref, mix_ref, prev, slot, flags, edge, x):
    """An output may differ from bf16(ref) by one bf16 ulp plus the f32 error of its operands, 2^-20 (|xn| + |prev|) scaled by the
    condition max(1, mean|x| / std(x)) of the rows its two LayerNorms came from: `bound` is the largest |out - bf16(ref)| / that
    allowance (<= 1), on plain and edge rows apart; `equal` is the share of outputs equal to bf16(ref) on plain rows.  `state` is
    max |state_out - LN| / max|LN| of the written slots, on edge rows divided by their condition."""
    got = pu.bf16_to_f32(out).astype(np.float64)
    want = pu.bf16_to_f32(pu.bf16_bits(mix_ref)).astype(np.float64)
    good = np.ones(x.shape[0], bool)
    good[edge] = False
    xd = x.astype(np.float64)
    cond = np.maximum(1.0, np.abs(xd).mean(axis=1) / np.maximum(xd.std(axis=1), 1e-300))
    cond_rows = np.maximum(cond, np.where(prev >= 0, cond[np.maximum(prev, 0)], 1.0))
    allow = bf16_ulp(want) + 2.0 ** -20 * cond_rows[None, :, None] * (np.abs(xn_ref) + np.abs(pv_ref))[None]
    ratio = np.abs(got - want) / allow
    plain = good & (np.where(prev >= 0, good[np.maximum(prev, 0)], True))
    m = dict(bound=ratio[:, plain].max(), equal=(got[:, plain] == want[:, plain]).mean(), edge_bound=ratio[:, ~plain].max(),
             state=0.0, state_edge=0.0)
    for r in np.nonzero(((flags & 1) != 0) & ((flags & 2) == 0))[0]:
        e = np.abs(so[slot[r]] - xn_ref[r]).max() / np.abs(xn_ref[r]).max()
        if good[r]:
            m["state"] = max(m["state"], e)
        else:
            m["state_edge"] = max(m["state_edge"], e / cond[r])
    return m


def ln_mix_run_case(ctx, Cw, nmix, in_place):
    """every form of one case: yields (form, form_used, metrics, unwritten slots kept bit for bit)"""
    rng = np.random.default_rng(Cw + nmix + 7 * in_place)
    x, lnw, lnb, mu, prev, slot, flags, state_in, edge = ln_mix_case(rng, Cw, nmix, in_place)
    xn_ref, pv_ref, mix_ref = ln_mix_ref(x, lnw, lnb, mu, prev, slot, state_in)
    sentinel = np.empty(state_in.shape, np.uint32)
    sentinel[:] = F32_SENTINEL
    sentinel = sentinel.view(np.float32)
    written = np.zeros(state_in.shape[0], bool)
    written[slot[((flags & 1) != 0) & ((flags & 2) == 0)]] = True
    keep = state_in if in_place else sentinel
    for form in ln_mix_forms(Cw):
        out, so, used = run_ln_mix(ctx, nmix, form, in_place, x, lnw, lnb, mu, prev, slot, flags, state_in, sentinel)
        kept = np.array_equal(so[~written].view(np.uint32), keep[~written].view(np.uint32))
        yield form, used, ln_mix_metrics(out, so, xn_ref, pv_ref, mix_ref, prev, slot, flags, edge, x), kept


LN_MIX_WIDTHS = (128, 192, 256, 512, 768, 1024)


def ln_mix_forms(Cw):
    return (0, 1) if Cw % 256 == 0 else (0,)


@pytest.mark.parametrize("in_place", [False, True], ids=["ping_pong", "in_place"])
@pytest.mark.parametrize("nmix", [1, 6])
@pytest.mark.parametrize("Cw", LN_MIX_WIDTHS)
def test_rwkv7_deep_ln_mix_vs_f64(gpu_ctx, Cw, nmix, in_place):
    """both kernel forms wherever the v8 one applies (they round the LayerNorm sums differently, so they are compared with the
    reference, not with each other); form 0 must pick v8 at every multiple of 256"""
    for form, used, m, kept in ln_mix_run_case(gpu_ctx, Cw, nmix, in_place):
        assert used == (8 if form == 0 and Cw % 256 == 0 else 1), (form, used)
        assert kept, "slots no row writes (flags bit 0 clear, or bit 1 set) must keep their contents bit for bit"
        assert m["bound"] <= 1.0 and m["equal"] >= 0.99 and m["edge_bound"] <= 1.0, (form, m)
        assert m["state"] <= 2.0 ** -20 and m["state_edge"] <= 2.0 ** -20, (form, m)


# ------------------------------------------------------------------------------------------------------------ model level
RWKV7_D256 = dict(RWKV7_TINY, d_model=256, n_heads=4, d_ffn=1024)


def load(ctx, cfg, W, engine=_lib.CZ_ENGINE_TCGEN05):
    model = cz.Model(ctx, cfg, engine=engine)
    for name, arr in W.items():
        model.set_tensor(name, arr)
    return model


def oracle_run(orc, targets, V):
    """logits[j] = the oracle's logits after BOS ++ the in-vocabulary targets[:j] (literal escapes do not step the model)"""
    cur = orc.step_logits(0)
    out = np.empty((len(targets), V), np.float32)
    for j, t in enumerate(targets):
        out[j] = cur
        if j + 1 < len(targets) and t < V:
            cur = orc.step_logits(int(t))
    return out


def deep_targets(V, n, seed, literal_share=0.0):
    rng = np.random.default_rng(seed)
    t = rng.integers(0, V, n).astype(np.uint32)
    lit = rng.random(n) < literal_share
    t[lit] = V + rng.integers(0, 256, int(lit.sum()))
    return t


def oracle_logits(cfg, W, targets, n_f32=None):
    """the bf16-rounding oracle over every position, the f32 oracle over the first n_f32 (default all)"""
    V = cfg["vocab"]
    w16 = oracle_run(oracle.Session.rwkv7(cfg, W, round_bf16=1), targets, V)
    w32 = oracle_run(oracle.Session.rwkv7(cfg, W, round_bf16=0), targets[: len(targets) if n_f32 is None else n_f32], V)
    return w16, w32


def parity(got, w16, w32):
    """per position: vs the bf16-rounding oracle, vs the f32 oracle, and the oracle against itself (the rounding points alone)"""
    n = len(w32)
    return pu.logits_parity(got, w16), pu.logits_parity(got[:n], w32), pu.logits_parity(w16[:n], w32)


def assert_parity(name, r, tols):
    """tols = (first 512 positions, positions from 512 on)"""
    assert r[:512].max() < tols[0], (name, int(r[:512].argmax()), float(r[:512].max()))
    assert len(r) <= 512 or r[512:].max() < tols[1], (name, 512 + int(r[512:].argmax()), float(r[512:].max()))


def deep_configs():
    """(name, cfg, weights builder, engines, n positions, literal share)"""
    return [
        ("RWKV7_TINY seed 7", RWKV7_TINY, lambda: make_weights(RWKV7_TINY, 7), (_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05), 4096, 0.05),
        ("long memory", RWKV7_TINY, lambda: long_memory(make_weights(RWKV7_TINY, 7), RWKV7_TINY), (_lib.CZ_ENGINE_TCGEN05,), 4096, 0.0),
        ("d_model 256", RWKV7_D256, lambda: make_weights(RWKV7_D256, 7), (_lib.CZ_ENGINE_TCGEN05,), 4096, 0.0),
    ]


FULL_CONFIG = ("0.1B shape", cz.RWKV7_0P1B, lambda: make_weights(cz.RWKV7_0P1B, 3), (_lib.CZ_ENGINE_TCGEN05,), 1024, 0.0)


@pytest.mark.parametrize("case", [0, 1, 2], ids=["seed7", "long_memory", "d256"])
def test_rwkv7_deep_tiny_every_position_vs_oracle(gpu_ctx, case):
    """every position of a 4,096-token BOS-started run (one of them with 5 % literal escapes, which do not step the model)"""
    name, cfg, mk, engines, n, lit = deep_configs()[case]
    W = mk()
    targets = deep_targets(cfg["vocab"], n, 40 + case, lit)
    t16, t32 = TOLS[name]
    w16, w32 = oracle_logits(cfg, W, targets)
    for eng in engines:
        model = load(gpu_ctx, cfg, W, eng)
        r16, r32, _ = parity(model.chunk_logits([0], targets), w16, w32)
        model.close()
        assert_parity((name, eng, "bf16 oracle"), r16, t16)
        assert_parity((name, eng, "f32 oracle"), r32, t32)


def test_rwkv7_deep_full_size_every_position_vs_oracle(gpu_ctx):
    """the 0.1B shape with make_weights (trained-like decay, LayerNorm and mix parameters, unlike random_init): every position of
    a 1,024-token run against both oracles"""
    name, cfg, mk, _, n, _ = FULL_CONFIG
    W = mk()
    targets = deep_targets(cfg["vocab"], n, 50)
    model = load(gpu_ctx, cfg, W)
    got = model.chunk_logits([0], targets)
    model.close()
    r16, r32, _ = parity(got, *oracle_logits(cfg, W, targets))
    assert_parity((name, "bf16 oracle"), r16, TOLS[name][0])
    assert_parity((name, "f32 oracle"), r32, TOLS[name][1])


NO_REPRIME = 1 << 40


def bits_per_token_case(ctx, cfg, W, head_scale, n, seed):
    """tokens drawn from the f32 oracle's own softmax (no reprime: RWKV-7 carries its state over the whole segment), so they cost
    far fewer than log2 V bits and the compressed size is sensitive to logits errors"""
    W = dict(W)
    W["lm_head.weight"] = bf16_exact(W["lm_head.weight"] * head_scale)
    orc = oracle.Session.rwkv7(cfg, W, round_bf16=0)
    ids = pu.sample_from_oracle(orc, n, np.random.default_rng(seed), context=NO_REPRIME, reprime_interval=NO_REPRIME)
    model = load(ctx, cfg, W)
    pays, seg = model.encode(ids, n_segments=1)
    ref, _ = oracle.Session.rwkv7(cfg, W, round_bf16=0).encode_tokens(np.concatenate([[0], ids]).astype(np.uint32), backend=1)
    assert np.array_equal(model.decode(pays, seg), ids)
    model.close()
    return len(pays[0]), len(ref), 8.0 * len(ref) / n, np.log2(cfg["vocab"])


def test_rwkv7_deep_tiny_bits_per_token_on_model_sampled_text(gpu_ctx):
    got, ref, bpt, log2v = bits_per_token_case(gpu_ctx, RWKV7_TINY, make_weights(RWKV7_TINY, 7), 2.0, 2000, 61)
    assert bpt < 0.6 * log2v, bpt
    assert abs(got - ref) <= 0.005 * ref, (got, ref)


def test_rwkv7_deep_full_size_bits_per_token_on_model_sampled_text(gpu_ctx):
    """make_weights text costs 13.2 of 16 bits per token, too flat for a size test; lm_head x 2 brings it to ~6"""
    got, ref, bpt, log2v = bits_per_token_case(gpu_ctx, cz.RWKV7_0P1B, make_weights(cz.RWKV7_0P1B, 3), 2.0, 1024, 62)
    assert bpt < 0.6 * log2v, bpt
    assert abs(got - ref) <= 0.005 * ref, (got, ref)
