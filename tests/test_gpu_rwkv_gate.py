"""Gated RWKV-7 streams end to end: hint primes with a history tail (`hist_take`) in the RWKV-7 decoder, its logits digests, the
gate's whole-history rule (max_context_length() = usize::MAX, src/models.rs:150) and `--reuse-scan-dir --backend rwkv7`."""
import os
import subprocess
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
from candlezip_b200 import _lib, container, gate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

pytestmark = pytest.mark.gpu
ENGINES = pytest.mark.parametrize("engine", [_lib.CZ_ENGINE_SIMT, _lib.CZ_ENGINE_TCGEN05], ids=["simt", "tc"])


def _rwkv_tiny(gpu_ctx, engine=_lib.CZ_ENGINE_TCGEN05):
    from rwkv7_weights import RWKV7_TINY, make_weights

    W = make_weights(RWKV7_TINY, 7)
    model = cz.Model(gpu_ctx, RWKV7_TINY, engine=engine)
    for name, arr in W.items():
        model.set_tensor(name, arr)
    return model, RWKV7_TINY, W


def _ids(rng, n, V, lit=0.1):
    ids = rng.integers(0, V, n).astype(np.uint32)
    mask = rng.random(n) < lit
    ids[mask] = V + rng.integers(0, 256, int(mask.sum()))  # literal escapes (src/main.rs:833-895)
    return ids


def host_prime(ids, i, hint, hist_take, V, bos=0):
    """the prime of a hist_take event, built from the known ids: the last hist_take symbols below V before i, BOS first when there
    are fewer, then the hint's tokens below V"""
    hist = [int(t) for t in ids[:i] if t < V]
    hist = hist[len(hist) - hist_take:] if hist_take <= len(hist) else [bos] + hist
    return np.array((hist if hist_take else []) + [int(t) for t in hint if t < V], np.uint32)


def _events(rng, n, V):
    """(i, hint, hold_until, hist_take): BOS-only history at i = 0, BOS padding with literals in the history and in the hint,
    an empty hint, events in consecutive agent chunks (128 tokens) and near the end"""
    hint = lambda k, lit=0.0: _ids(rng, k, V, lit)  # noqa: E731
    return [(0, hint(7), 64, 5), (40, hint(12, 0.4), 104, 100), (200, np.zeros(0, np.uint32), 264, 30), (383, hint(25), 447, 150),
            (511, hint(9, 0.2), 575, 400), (n - 4, hint(6), n + 60, 50), (n - 1, hint(3), n + 63, 2)]


def _units(ids, events, V):
    """(prime, first, end) of every unit of the stream: BOS until the first event, then each event's prime"""
    cuts = [(0, np.array([0], np.uint32))] if events[0][0] != 0 else []
    cuts += [(i, host_prime(ids, i, h, ht, V)) for i, h, _, ht in events]
    return [(p, a, cuts[k + 1][0] if k + 1 < len(cuts) else len(ids)) for k, (a, p) in enumerate(cuts)]


def _gpu_logits_payload(model, ids, events, V):
    """oracle coder on the GPU's own logits of every unit (chunk_logits), literal alphabet"""
    logits = np.concatenate([model.chunk_logits(p, ids[a:b]) for p, a, b in _units(ids, events, V)])
    bounds = [tuple(int(x) for x in oracle.logits_to_cdf(logits[j], 1)[[ids[j], ids[j] + 1]]) for j in range(len(ids))]
    return oracle.ac_encode(bounds), logits


@ENGINES
def test_hist_take_round_trip_equals_explicit_primes_and_oracle(gpu_ctx, engine):
    model, cfg, W = _rwkv_tiny(gpu_ctx, engine)
    V = cfg["vocab"]
    rng = np.random.default_rng(2024)
    n = 900
    ids = _ids(rng, n, V)
    events = _events(rng, n, V)
    assert sum(1 for t in ids[:40] if t < V) < 100  # the second event pads with BOS
    pays, seg = model.encode(ids, n_segments=1, events=events)
    assert np.array_equal(model.decode(pays, seg, events=events), ids)
    # the same stream from primes built on the host (hist_take = 0)
    explicit = [(i, host_prime(ids, i, h, ht, V), hold, 0) for i, h, hold, ht in events]
    px, _ = model.encode(ids, n_segments=1, events=explicit)
    assert px == pays
    assert np.array_equal(model.decode(px, seg, events=explicit), ids)
    # bit-exact: the oracle coder fed with the GPU's own logits of every unit
    want, _ = _gpu_logits_payload(model, ids, events, V)
    assert want == pays[0]
    # size: the f32 oracle running the reference loop with the same primes
    if engine == _lib.CZ_ENGINE_TCGEN05:
        orc = oracle.Session.rwkv7(cfg, W)
        ref, _ = orc.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32), backend=1, events=[e[:3] for e in explicit])
        assert abs(len(pays[0]) - len(ref)) <= 0.005 * len(ref) + 2, (len(pays[0]), len(ref))


@ENGINES
def test_long_prime_in_slabs(gpu_ctx, engine):
    """a prime of the whole history (the gate's rule on RWKV-7) spans several of the decoder's prime slabs: same payload as the
    explicit prime coded in one slab, and the same ids back whatever the slab size"""
    model, cfg, _ = _rwkv_tiny(gpu_ctx, engine)
    V = cfg["vocab"]
    rng = np.random.default_rng(99)
    n = 800
    ids = _ids(rng, n, V, 0.05)
    hint = _ids(rng, 30, V, 0.1)
    events = [(300, hint[:10], 364, 301), (700, hint, 764, 701)]
    prime = host_prime(ids, 700, hint, 701, V)
    assert len(prime) >= 3 * 128 + 1
    explicit = [(i, host_prime(ids, i, h, ht, V), hold, 0) for i, h, hold, ht in events]
    px, seg = model.encode(ids, n_segments=1, events=explicit)
    pays, _ = model.encode(ids, n_segments=1, events=events, max_batch_tokens=128)
    assert pays == px
    want, _ = _gpu_logits_payload(model, ids, events, V)
    assert want == pays[0]
    for rows in (128, 100, 0):  # 0: the default slab
        assert np.array_equal(model.decode(pays, seg, events=events, max_batch_tokens=rows), ids), rows


def test_empty_prime_is_invalid_on_both_sides(gpu_ctx):
    model, cfg, _ = _rwkv_tiny(gpu_ctx)
    V = cfg["vocab"]
    ids = np.arange(50, dtype=np.uint32) % V
    bad = [(10, np.array([V + 3], np.uint32), 74, 0)]  # only a literal escape, no history
    for call in (lambda: model.encode(ids, events=bad), lambda: model.decode([b"\0" * 8], np.array([0, 50], np.uint64), events=bad)):
        with pytest.raises(_lib.CzError) as e:
            call()
        assert e.value.code == _lib.CZ_ERR_INVALID


def _b3(col):
    return np.frombuffer(container.blake3_16(np.ascontiguousarray(col, np.float32).tobytes()), np.uint8)


@ENGINES
def test_decode_digests_equal_encode_digests(gpu_ctx, engine):
    model, cfg, _ = _rwkv_tiny(gpu_ctx, engine)
    V = cfg["vocab"]
    rng = np.random.default_rng(5)
    n = 900
    ids = _ids(rng, n, V, 0.15)
    ids[100:104] = V + 65  # consecutive literals share one logits column
    events = _events(rng, n, V)
    dig = model.watch_digests(n)
    try:
        pays, seg = model.encode(ids, n_segments=1, events=events)
        enc = dig.copy()
        assert not np.any(np.all(enc == 0, axis=1))
        for j in (101, 102, 103, 104):  # literals do not step: the run and the symbol after it are coded from index 100's column
            assert np.array_equal(enc[j], enc[100]), j
        _, logits = _gpu_logits_payload(model, ids, events, V)
        for j in (0, 1, 39, 40, 99, 101, 200, 511, n - 4, n - 1):
            assert np.array_equal(enc[j], _b3(logits[j])), j
        dig[:] = 0
        assert np.array_equal(model.decode(pays, seg, events=events), ids)
        assert np.array_equal(dig, enc), "decode digests differ from encode digests"
        # several segments, no events: the lock-step decoder digests every live stream
        p3, s3 = model.encode(ids, n_segments=3)
        enc3 = dig.copy()
        dig[:] = 0
        assert np.array_equal(model.decode(p3, s3), ids) and np.array_equal(dig, enc3)
    finally:
        model.watch_digests(0)


def test_gate_scan_whole_history_and_round_trip(gpu_ctx):
    model, cfg, W = _rwkv_tiny(gpu_ctx)
    V = cfg["vocab"]
    rng = np.random.default_rng(77)
    n = 1000
    ids = _ids(rng, n, V, 0.05)
    tok = lambda s, m: [(ord(ch) * 7) % V for ch in s][:m]  # noqa: E731
    texts = {1: "Alpha Beta 12 gamma " * 9, 2: "", 3: "Delta 7 Epsilon " * 30}
    assert gate.max_ctx_for(model) == gate.MAX_CTX_RWKV7
    pays, seg, records, rows, events = gate.scan_encode(model, ids, texts, tok, agent_chunk=256, scan_lookahead=200)
    assert len(records) == 3 and all(ht == i + 1 for i, _, _, ht in events)
    hints = [[np.asarray(tok(c, 512), np.uint32) for c in gate.build_candidates(texts.get(k + 1, ""))] for k in range(len(records))]
    dec = gate.events_from_records(records, hints, 256, n, scan_lookahead=200, max_ctx=gate.MAX_CTX_RWKV7)
    assert len(dec) == len(events) and all(a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:] for a, b in zip(dec, events))
    assert np.array_equal(model.decode(pays, seg, events=dec or None), ids)
    # every boundary gated (whatever the random weights decide): the whole history plus the whole hint
    forced = [1 | (0 << 1) | (bid << 3) for bid in (3, 1, 0)]
    fev = gate.events_from_records(forced, hints, 256, n, scan_lookahead=200, max_ctx=gate.MAX_CTX_RWKV7)
    assert [e[0] for e in fev] == [255, 511, 767] and [len(e[1]) for e in fev] == [len(h[0]) for h in hints]
    fp, fs = model.encode(ids, n_segments=1, events=fev)
    assert np.array_equal(model.decode(fp, fs, events=fev), ids)
    # the scan: identical conditioned jobs share one stream; one job against the oracle with the whole history
    jobs, plan = gate.plan_scan(ids, texts, tok, 256, 200, max_ctx=gate.MAX_CTX_RWKV7)
    assert len(jobs) == len(plan) + sum(len({h.tobytes() for h in e["hints"] if len(h)}) for e in plan) < len(plan) + 8
    bits = model.xe_bits(jobs)
    seq = np.concatenate([[0], ids]).astype(np.uint32)
    orc = oracle.Session.rwkv7(cfg, W, round_bf16=1)
    e = plan[2]
    i, slot = e["i"], e["slots"][0 * 4 + 2]
    assert slot == e["slots"][0] == e["slots"][1] == e["slots"][3] == e["slots"][4]  # four budgets; candidates 0 and 1 are one text
    want = orc.xe_bits(seq[:i], seq[i:i + 200], e["hints"][0], backend=1)
    assert abs(bits[slot] - want) <= 0.01 * want, (bits[slot], want)


def _cli(*args, timeout=900):
    return subprocess.run([sys.executable, "-m", "candlezip_b200", *args], cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_cli_rwkv7_gate_replay(gpu_ctx, tmp_path):
    """`self-test --backend rwkv7 --reuse-scan-dir` and `compress` / `decompress` as separate processes"""
    import json

    import corpus

    data = corpus.load("alice29.txt")[:2600]
    src = tmp_path / "alice_head.txt"
    src.write_bytes(data)
    rdir = tmp_path / "run"
    rdir.mkdir()
    with open(rdir / "agent_cache.jsonl", "w", encoding="utf-8") as f:
        f.write(json.dumps({"chunk_index": 1, "agent_text": data[512:1400].decode("latin-1"), "agent_calls": 3}) + "\n")
        f.write(json.dumps({"chunk_index": 3, "agent_text": "Alice 1865 Rabbit-Hole\nDown the 2nd well", "agent_calls": 1}) + "\n")
    out_dir = tmp_path / "scan_out"
    common = ["--backend", "rwkv7", "--reuse-scan-dir", str(rdir), "--scan-lookahead", "300"]
    r = _cli("self-test", str(src), *common, "--scan-output-dir", str(out_dir))
    assert r.returncode == 0 and "roundtrip OK" in r.stdout and "scan: 5 boundaries" in r.stdout, (r.stdout, r.stderr[-800:])
    rows = open(out_dir / "proof.csv").read().strip().split("\n")
    assert len(rows) == 6 and rows[0].startswith("file,chunk_index,start_token,end_token,agent_text_len")
    blob = tmp_path / "a.canz"
    r = _cli("compress", str(src), str(blob), *common)
    assert r.returncode == 0, r.stderr[-800:]
    f, _, gates, _, _, _ = container.read_container(blob.read_bytes())
    assert gates is not None and len(gates) == 5 and f["vocab_size"] == cz.RWKV7_0P1B["vocab"]
    back = tmp_path / "a.out"
    r = _cli("decompress", str(blob), str(back), *common)
    assert r.returncode == 0, r.stderr[-800:]
    assert back.read_bytes() == data
