"""GPU suite, round-2 additions: id validation (no out-of-bounds embedding reads), the lock-step decoder's precondition,
on-GPU logits digests, the sharded product path and the replayed agentic gate."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import candlezip_b200 as cz
import oracle
from candlezip_b200 import _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def _tiny(gpu_ctx, seed=5, embed_std=0.05, engine=_lib.CZ_ENGINE_TCGEN05):
    return cz.Model(gpu_ctx, cz.SMOLLM_TINY, engine=engine).random_init(seed, 0.05, embed_std)


def test_out_of_range_ids_are_rejected_everywhere(gpu_ctx):
    """ADVICE r1: an id >= vocab used to index the embedding table out of bounds.  Host-side ids are rejected before any launch
    (CZ_ERR_SYMBOL_RANGE naming the index); ids that exist only on the device are caught by the kernels; the ctx stays usable."""
    model = _tiny(gpu_ctx)
    V = 1024
    rng = np.random.default_rng(0)
    ids = rng.integers(0, V, 700).astype(np.uint32)
    good, _ = model.encode(ids)

    def rejects(fn):
        with pytest.raises(cz.CzError) as e:
            fn()
        assert e.value.code == _lib.CZ_ERR_SYMBOL_RANGE, e.value

    bad = ids.copy()
    bad[123] = V
    rejects(lambda: model.encode(bad))
    rejects(lambda: model.encode(ids, bos=V + 5))
    rejects(lambda: model.encode(ids, events=[(100, np.array([1, 2, 1 << 30], np.uint32), 200)]))
    rejects(lambda: model.decode(good, [0, 700], bos=4000))
    rejects(lambda: model.xe_bits([(np.array([3, V], np.uint32), ids[:5])]))
    rejects(lambda: model.xe_bits([(ids[:9], np.array([3, 70000], np.uint32))]))
    rejects(lambda: model.chunk_logits(np.array([0xFFFFFFFF], np.uint32), ids[:3]))
    s = model.session()
    rejects(lambda: s.step_logits_tensor(V))
    rejects(lambda: s.reprime_with_history_and_get_last_logits_tensor(np.array([1, 2, V + 1], np.uint32)))
    # device-resident ids: only the kernels can see them
    import torch

    n = len(bad)
    seg = cz.split_segments(n, 1)
    sched, keep = model._schedule(n, seg, 0, 512, 512, None, 0)
    d_ids = torch.from_numpy(bad.astype(np.int64)).to(torch.int32).cuda()
    out = torch.empty(4 * n + 64, dtype=torch.uint8, device="cuda")
    off = np.zeros(2, np.uint64)
    rc = _lib.lib.cz_encode_dev(model._h, C.c_void_p(d_ids.data_ptr()), n, C.byref(sched), C.c_void_p(out.data_ptr()), 4 * n + 64,
                                off.ctypes.data_as(_lib.u64p))
    assert rc == _lib.CZ_ERR_SYMBOL_RANGE, (rc, _lib.lib.cz_last_error())
    # nothing was poisoned: the same model still produces the same bytes
    again, _ = model.encode(ids)
    assert again == good
    # RWKV-7: literal escapes (V .. V+255) are part of the coded alphabet, anything above is not
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from rwkv7_weights import RWKV7_TINY, make_weights

    rm = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        rm.set_tensor(name, arr)
    rv = RWKV7_TINY["vocab"]
    rid = rng.integers(0, rv, 50).astype(np.uint32)
    rid[7] = rv + 255
    rm.encode(rid)
    rid[7] = rv + 256
    rejects(lambda: rm.encode(rid))


def test_decode_requires_non_increasing_segments(gpu_ctx):
    """the lock-step decoder's documented precondition (include/candlezip_b200.h, cz_decode): longest segments first"""
    model = _tiny(gpu_ctx)
    ids = np.random.default_rng(1).integers(0, 1024, 900).astype(np.uint32)
    seg = np.array([0, 200, 900], np.uint64)  # 200 then 700 tokens: increasing
    pays, _ = model.encode(ids, seg_start=seg)  # the encoder has no such restriction
    with pytest.raises(cz.CzError) as e:
        model.decode(pays, seg)
    assert e.value.code == _lib.CZ_ERR_UNSUPPORTED and "non-increasing" in str(e.value)
    ok = np.array([0, 700, 900], np.uint64)
    pays, _ = model.encode(ids, seg_start=ok)
    assert np.array_equal(model.decode(pays, ok), ids)


def _b3(a):
    from candlezip_b200 import container

    raw = np.ascontiguousarray(a, np.float32).tobytes()
    d = container.blake3_16(raw)  # the host implementation, itself pinned to the `blake3` package in the CPU suite
    try:
        import blake3

        assert blake3.blake3(raw).digest()[:16] == d
    except ImportError:
        pass
    return np.frombuffer(d, np.uint8)


def test_logits_digests_on_gpu_match_blake3_and_audit_decode(gpu_ctx):
    """SURVEY 8 f-4: blake3_f32_bin16 per step (src/main.rs:955-961, 2328-2342) computed on the GPU: equal to BLAKE3-128 of the same
    logits bytes on the host, identical for every wave size, and the decoder's digests equal the encoder's (the watchdog's
    enc/dec comparison, src/main.rs:2629-2647, as a determinism audit)."""
    model = _tiny(gpu_ctx)
    rng = np.random.default_rng(3)
    n = 1700
    ids = rng.integers(0, 1024, n).astype(np.uint32)
    dig = model.watch_digests(n)
    pays, seg = model.encode(ids, n_segments=3)
    enc = dig.copy()
    # every position hashed, none left zero; only the three segments' first positions (BOS alone) share their logits
    assert len(np.unique(enc, axis=0)) == n - 2 and np.array_equal(enc[int(seg[0])], enc[int(seg[1])])
    # segment 0, chunk 0 (BOS + up to 512 tokens) and its second chunk (511-token prime): digests of the very logits that were coded
    a, b = int(seg[0]), int(seg[1])
    logits = model.chunk_logits([0], ids[a:a + 512])
    for j in (0, 1, 255, 511):
        assert np.array_equal(enc[a + j], _b3(logits[j])), j
    seq = np.concatenate([[0], ids[a:b]]).astype(np.uint32)
    l2 = model.chunk_logits(seq[2:513], ids[a + 512:b])
    for j in (0, 17, b - a - 513):
        assert np.array_equal(enc[a + 512 + j], _b3(l2[j])), j
    dig[:] = 0
    model.encode(ids, n_segments=3, max_batch_tokens=700)  # other wave boundaries, same digests
    assert np.array_equal(dig, enc)
    dig[:] = 0
    out = model.decode(pays, seg)
    assert np.array_equal(out, ids) and np.array_equal(dig, enc), "decode digests differ from encode digests"
    model.watch_digests(0)
    # V = 4099 is not a multiple of the 64-byte block or the 1 KiB chunk: partial last block / chunk, odd tree shape
    cfg = dict(cz.SMOLLM_TINY, vocab=4099)
    m2 = cz.Model(gpu_ctx, cfg).random_init(9, 0.05, 0.05)
    ids2 = rng.integers(0, 4099, 40).astype(np.uint32)
    d2 = m2.watch_digests(40)
    m2.encode(ids2)
    lg = m2.chunk_logits([0], ids2)
    for j in (0, 39):
        assert np.array_equal(d2[j], _b3(lg[j])), j


def test_logits_digests_full_size_and_rwkv(gpu_ctx):
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    rng = np.random.default_rng(4)
    ids = rng.integers(0, 256, 1300).astype(np.uint32)
    dig = model.watch_digests(len(ids))
    pays, seg = model.encode(ids, n_segments=2)
    enc = dig.copy()
    lg = model.chunk_logits([0], ids[:3])
    assert np.array_equal(enc[0], _b3(lg[0])) and np.array_equal(enc[2], _b3(lg[2]))  # 192 chunks: the 128 + 64 tree
    dig[:] = 0
    assert np.array_equal(model.decode(pays, seg), ids) and np.array_equal(dig, enc)
    model.close()
    from rwkv7_weights import RWKV7_TINY, make_weights

    rm = cz.Model(gpu_ctx, RWKV7_TINY)
    for name, arr in make_weights(RWKV7_TINY, 7).items():
        rm.set_tensor(name, arr)
    V = RWKV7_TINY["vocab"]
    rid = rng.integers(0, V, 300).astype(np.uint32)
    rid[rng.random(300) < 0.1] = V + 9  # literal escapes are coded from the same logits but do not step the model
    rd = rm.watch_digests(300)
    rm.encode(rid)
    rl = rm.chunk_logits([0], rid)
    for j in (0, 1, 150, 299):
        assert np.array_equal(rd[j], _b3(rl[j])), j


def _hint_tok(vocab):
    import corpus

    m = corpus.spread_map(vocab)
    return lambda text, max_tokens: m[np.frombuffer(text.encode("utf-8"), np.uint8)][:max_tokens]


def test_config4_replay_of_the_shipped_asyoulik_run(gpu_ctx, fixtures, tmp_path):
    """BASELINE config 4 on the reference's own artefacts: the shipped SmolLM2 token ids of asyoulik.txt (39,915 ids from
    watchdog_decode_steps.jsonl) + the shipped agent_cache.jsonl / proof.csv (results_300s_nomem/asyoulik_*), replayed without
    an agent (`--reuse-scan-dir`, src/main.rs:1966-1978, loaders :1152-1195).
      (a) cached mode (:2221-2268): the ledger's (gate, candidate, budget) are applied as-is -> AGT2 records == the proof.csv
          columns for all 77 boundaries; the gated stream round-trips (prefix) from (records, agent texts) alone;
      (b) rescan mode (:2043-2072): all baseline / hint-conditioned XE passes of all boundaries as ONE batch of paired streams,
          a proof.csv written in the reference's 26-column format whose structural columns equal the shipped ledger's.
    The agent texts are tokenised byte-level (no tokenizer.json offline) and the weights are random-init, so the XE columns are
    not comparable with the shipped ones -- only their bookkeeping is."""
    import corpus
    from candlezip_b200 import container, gate

    ids = fixtures["run_asyoulik_syms"].astype(np.uint32)
    assert len(ids) == 39915 and ids.max() < 49152
    texts, calls, decisions, shipped = gate.load_replay(corpus.replay("asyoulik"))
    assert len(shipped) == 77 and len(texts) == 30 == sum(g for g, _, _ in decisions.values())
    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    tok = _hint_tok(49152)
    # ---- (a) cached decisions ----
    records, events = gate.events_from_decisions(ids, texts, decisions, tok, agent_chunk=512)
    want = fixtures["run_asyoulik_gates"]  # [chunk_index, gate, candidate, budget] per proof.csv row
    assert len(records) == 77 and [(r & 1, (r >> 1) & 3, (r >> 3) & 3) for r in records] == [tuple(int(x) for x in w[1:]) for w in want]
    assert len(events) == 30 and all(len(h) > 0 for _, h, _, _ in events)
    pays, seg = model.encode(ids, n_segments=1, events=events)
    plain, _ = model.encode(ids, n_segments=1)
    assert pays != plain
    blob = container.write_container(dict(token_count=len(ids), orig_len_bytes=125179, vocab_size=49152,
                                          reserved_flags=int(_lib.lib.cz_flags_pack(1, 0, 1, 512))), b"model.safetensors", pays, gates=records)
    f, _, g2, _, _, p2 = container.read_container(blob)
    assert g2 == records and p2 == pays and (f["reserved_flags"] >> 16) == 512
    # decode side: records + the same agent texts rebuild the events (main.rs:2545-2614); round trip of a 6-boundary prefix
    n_pre = 3300
    rec_pre, ev_pre = gate.events_from_decisions(ids[:n_pre], texts, decisions, tok, agent_chunk=512)
    pp, sp = model.encode(ids[:n_pre], n_segments=1, events=ev_pre)
    hints = [[np.asarray(tok(c, 512), np.uint32) for c in gate.build_candidates(texts.get(k + 1, ""))] for k in range(len(rec_pre))]
    dec_events = gate.events_from_records(rec_pre, hints, 512, n_pre)
    assert len(dec_events) == len(ev_pre) and all(a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2:] == b[2:] for a, b in zip(dec_events, ev_pre))
    assert np.array_equal(model.decode(pp, sp, events=dec_events), ids[:n_pre])
    # ---- (b) rescan: paired streams, ledger ----
    pays2, seg2, records2, rows, events2 = gate.scan_encode(model, ids, texts, tok, agent_chunk=512, scan_lookahead=512)
    assert len(rows) == 77 and [r["chunk_index"] for r in rows] == list(range(1, 78))
    led = gate.ledger_rows(rows, "final_bench/cantrbry/asyoulik.txt", texts, calls, agent_chunk=512, domain="cantrbry")
    path = tmp_path / "proof.csv"
    gate.write_proof_csv(str(path), led)
    t2, c2, d2, back = gate.load_replay(str(tmp_path))  # the written ledger parses with the reference's own loader rules
    assert len(back) == 77 and all(len(r) == 26 for r in back)
    for mine, ref in zip(back, shipped):
        assert mine[1:4] == ref[1:4]                                  # chunk_index, start_token, end_token
        ci = int(ref[1])
        if ci in texts:                                               # the cache holds the texts of the gated chunks only
            assert mine[4] == ref[4] and mine[10] == ref[10]          # agent_text_len, agent_calls
            assert mine[19] == ref[19] == mine[20]                    # args_hash = output_hash = BLAKE3-128 of the agent text
        assert mine[25] == ref[25]                                    # chunk_id "asyoulik:<k>"
        assert float(mine[6]) > 0 and abs(float(mine[6]) - float(mine[7]) - float(mine[8])) < 1e-5
    assert all(r["gate"] == 0 and r["bits_saved"] == 0.0 for r in rows if r["chunk_index"] not in texts)  # empty hints never gate


_SHARD_WORKER = r"""
import os, sys
import numpy as np
ROOT = sys.argv[1]
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")]
import torch.distributed as dist
import candlezip_b200 as cz
from candlezip_b200 import container, sharding
import corpus
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{os.environ['CZ_PORT']}", rank=rank, world_size=world)
model = cz.Model(cz.Context(rank), cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
data = corpus.load("enwik8_3mib")[:40000]
ids = corpus.byte_ids(data, 49152, True)
pays, seg = sharding.encode_sharded(lambda part, s: model.encode(part, seg_start=s)[0], ids, 10, rank, world, dist)
blob = None
if rank == 0:
    f = dict(token_count=len(ids), orig_len_bytes=len(data), vocab_size=49152, orig_hash16=container.blake3_16(data))
    blob = container.write_container(f, b"random-init", pays, seg_tokens=np.diff(seg))
lst = [blob]
dist.broadcast_object_list(lst, src=0)
_, _, _, _, st, payloads = container.read_container(lst[0])
seg2 = np.concatenate([[0], np.cumsum(st)]).astype(np.uint64)
out = sharding.decode_sharded(lambda p, s: model.decode(p, s), payloads, seg2, rank, world, dist)
if rank == 0:
    assert corpus.ids_to_bytes(out, 49152, True) == data
    open(sys.argv[2], "wb").write(lst[0])
dist.destroy_process_group()
"""


def test_sharded_product_path_on_two_gpus_gives_identical_container(gpu_ctx, tmp_path):
    """SURVEY 8e on hardware: ONE input through candlezip_b200.sharding on 2 GPUs (contiguous segment ranges per rank,
    Model.encode / Model.decode on each, gather to rank 0, container assembly) == the single-GPU container, byte for byte.
    Skips cleanly on a 1-GPU box (bench.py --gpus N prints the same check as `sharded.container_blake3_16` for N = 1/2/4/8)."""
    import socket
    import subprocess

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import corpus
    from candlezip_b200 import container

    model = cz.Model(gpu_ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    data = corpus.load("enwik8_3mib")[:40000]
    ids = corpus.byte_ids(data, 49152, True)
    pays, seg = model.encode(ids, n_segments=10)
    f = dict(token_count=len(ids), orig_len_bytes=len(data), vocab_size=49152, orig_hash16=container.blake3_16(data))
    single = container.write_container(f, b"random-init", pays, seg_tokens=np.diff(seg))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(_SHARD_WORKER)
    outp = tmp_path / "two_gpu.canz"
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(outp)],
                              env=dict(os.environ, RANK=str(r), WORLD_SIZE="2", CZ_PORT=str(port)), stderr=subprocess.PIPE)
             for r in range(2)]
    for p in procs:
        _, err = p.communicate(timeout=600)
        assert p.returncode == 0, err.decode()[-800:]
    assert outp.read_bytes() == single


def test_zero_width_symbol_falls_back_to_a_stored_container(gpu_ctx):
    """ADVICE r1 (low): SmolLM coding has no probability floor; a peaky model meets tokens of mass < 2^-30 on surprising input.
    cz_encode reports CZ_ERR_ZERO_WIDTH with the token index (the reference would silently corrupt the stream); the file-level
    compress() then stores the bytes uncoded under CZ_FLAG_STORED so that decode(encode(x)) == x still holds."""
    from candlezip_b200 import codec, container

    model = cz.Model(gpu_ctx, cz.SMOLLM_TINY).random_init(5, 0.05, 1.5)  # very peaky logits (std ~ 20)
    data = bytes(np.random.default_rng(0).integers(0, 256, 3000, dtype=np.uint8))
    with pytest.raises(cz.CzError) as e:
        model.encode(np.frombuffer(data, np.uint8).astype(np.uint32))
    assert e.value.code == _lib.CZ_ERR_ZERO_WIDTH and "coded index" in str(e.value)
    blob = codec.compress(model, data)
    f = container.read_container(blob)[0]
    assert f["reserved_flags"] & _lib.CZ_FLAG_STORED and f["orig_len_bytes"] == len(data)
    assert codec.decompress(model, blob) == data
    bad = bytearray(blob)
    bad[-1] ^= 1
    with pytest.raises(ValueError):
        codec.decompress(model, bytes(bad))


def test_cdf_fast_paths_equal_the_originals_exhaustively(gpu_ctx):
    """csrc/cdf_fast.cuh: (1) expf through integer conversions == expf through F2F conversions for EVERY argument the fast path
    accepts (all 2^31 non-negative f32 patterns are visited), and the device expf's checksum over the whole domain equals the
    oracle's (whose expf is verified exhaustively against the host glibc expf, the one Rust's f32::exp calls, src/main.rs:791);
    (2) the reciprocal-based division (Markstein) == IEEE division on 2^34 random operand pairs."""
    bad, chk, first = C.c_uint64(), C.c_uint64(), C.c_uint64()
    _lib.check(_lib.lib.cz_test_expf_exhaustive(gpu_ctx._h, C.byref(bad), C.byref(chk), C.byref(first)))
    assert bad.value == 0, f"{bad.value} arguments differ, first bit pattern {first.value:#x}"
    assert chk.value == oracle.lib.czo_expf_checksum(0, 1 << 31)
    for seed in (1, 2):
        m = C.c_uint64()
        _lib.check(_lib.lib.cz_test_div_random(gpu_ctx._h, seed, 1 << 33, C.byref(m)))
        assert m.value == 0, m.value


@pytest.mark.parametrize("m", [40, 260, 261, 1024, 1027])
@pytest.mark.parametrize("mode", [0, 1])
def test_cdf_bounds_and_xe_tma_and_direct_stats_kernels(gpu_ctx, mode, m):
    """the round-2 stats / sorted-prefix / XE kernels against the oracle on m columns (ld = m): 260 and 1024 take the TMA-staged
    full passes, 40 (too few columns) and the odd counts (ld % 4 != 0) the direct-load kernel; with symbols at both ends of the
    alphabet, literal escapes, logits more than 87 below the maximum (the conversion fallback), -inf entries and exact ties; then
    (once) a model-level encode whose ragged column counts go through the same kernels, checked against the oracle coder on the
    GPU's own logits."""
    import test_gpu_parity as tgp

    rng = np.random.default_rng([100 + mode, m])
    v = 2309 if mode else 2304
    n_sym = v + 256 if mode else v
    logits = tgp._adversarial_logits(rng, v, m)
    logits[:, m // 2] = rng.normal(0, 30, v)      # most entries > 87 below the max: slow conversion path, tiny / zero terms
    syms = rng.integers(0, n_sym, m).astype(np.uint32)
    syms[:6] = [0, n_sym - 1, 1, v - 1, min(v, n_sym - 1), n_sym - 2]
    lo, hi = gpu_ctx.cdf_bounds(logits, syms, mode)
    xe = gpu_ctx.xe_bits_cols(logits, syms, mode)
    for j in range(m):
        cdf = oracle.logits_to_cdf(logits[:, j], mode)
        assert (int(lo[j]), int(hi[j])) == (int(cdf[syms[j]]), int(cdf[syms[j] + 1])), (m, j, syms[j])
        pdf = oracle.combined_pdf_with_literals(logits[:, j]) if mode else oracle.softmax_pdf_floor(logits[:, j])
        want = -np.log2(max(pdf[syms[j]], 1e-300))
        assert abs(xe[j] - want) <= 1e-12 * max(1.0, abs(want)), (m, j)
    if mode == 0 and m == 40:
        model = _tiny(gpu_ctx)
        ids = rng.integers(0, 1024, 701).astype(np.uint32)
        pays, seg = model.encode(ids, n_segments=1)
        lg = np.concatenate([model.chunk_logits([0], ids[:512]), model.chunk_logits(np.concatenate([[0], ids])[2:513], ids[512:])])
        bounds = [tuple(int(x) for x in oracle.logits_to_cdf(lg[j], 0)[[ids[j], ids[j] + 1]]) for j in range(701)]
        assert oracle.ac_encode(bounds) == pays[0]


@pytest.mark.parametrize("mode", [0, 1])
def test_cdf_prefix_walk_through_the_ecache_and_its_fallback(gpu_ctx, mode):
    """csrc/cdf_kernels.cu (e-cache): the stats pass leaves e_v, v <= coded symbol, contiguously per column and the prefix walk reads
    that instead of the vocab-major logits.  Same bounds as the oracle (src/main.rs:784-824 / 758-782) (a) through the cache
    (heavy-tailed symbols at the default capacity; uniform symbols with the capacity raised to the whole batch), (b) when the batch
    does not fit (uniform symbols at the default capacity: the flag computed on the device sends the walk back to the logits) and
    (c) with the cache disabled; the state hook says which of the three ran."""
    import test_gpu_parity as tgp

    def state():
        st, g = C.c_int(), C.c_uint64()
        _lib.check(_lib.lib.cz_test_cdf_ecache_state(gpu_ctx._h, C.byref(st), C.byref(g)))
        return st.value, g.value

    rng = np.random.default_rng(300 + mode)
    v = 2309 if mode else 2304  # (2309: a ragged last 16-row tile and a ragged last cache group)
    n_sym = v + 256 if mode else v
    try:
        for m in (260, 1031 // 4 * 4, 2048):
            logits = tgp._adversarial_logits(rng, v, m)
            logits[:, m // 3] = rng.normal(0, 30, v)  # entries > 87 below the max: the conversion path inside a cached column
            heavy = np.minimum((rng.random(m) ** 6 * n_sym).astype(np.uint32), n_sym - 1)  # mean id / alphabet = 1/7
            heavy[:8] = [0, 1, 7, 8, 9, v - 1, min(v, n_sym - 1), n_sym - 1]
            heavy[m // 3] = v - 2
            uniform = rng.integers(0, n_sym, m).astype(np.uint32)
            want = {}
            for name, syms in (("heavy", heavy), ("uniform", uniform)):
                cdfs = [oracle.logits_to_cdf(logits[:, j], mode) for j in range(m)]
                want[name] = (np.array([c[s] for c, s in zip(cdfs, syms)], np.uint32), np.array([c[s + 1] for c, s in zip(cdfs, syms)], np.uint32))
            runs = [("heavy", None, 1), ("uniform", None, 0), ("uniform", "1.0", 1), ("heavy", "off", -1)]
            for name, frac, expect in runs:
                os.environ.pop("CZ_CDF_ECACHE_FRAC", None)
                os.environ.pop("CZ_CDF_NO_ECACHE", None)
                if frac == "off":
                    os.environ["CZ_CDF_NO_ECACHE"] = "1"
                elif frac:
                    os.environ["CZ_CDF_ECACHE_FRAC"] = frac
                syms = heavy if name == "heavy" else uniform
                lo, hi = gpu_ctx.cdf_bounds(logits, syms, mode)
                st, groups = state()
                assert st == expect, (m, name, frac, st, groups)
                if st == 1:
                    need = sum((min(int(x) + 1, v) + 7) // 8 for x in syms)
                    assert groups == need, (groups, need)
                assert np.array_equal(lo, want[name][0]) and np.array_equal(hi, want[name][1]), (m, name, frac)
    finally:
        os.environ.pop("CZ_CDF_ECACHE_FRAC", None)
        os.environ.pop("CZ_CDF_NO_ECACHE", None)


def test_cli_twin_gate_scan_replay_self_test(gpu_ctx, tmp_path):
    """`python -m candlezip_b200 self-test FILE --reuse-scan-dir DIR` (src/main.rs:156-221 with --reuse-scan-dir, :1966-1978): the gate
    scan replayed from an agent_cache.jsonl in the reference's format; AGT2 container, proof.csv ledger, byte-exact round trip."""
    import json
    import subprocess

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
    r = subprocess.run([sys.executable, "-m", "candlezip_b200", "self-test", str(src), "--reuse-scan-dir", str(rdir), "--scan-output-dir", str(out_dir),
                        "--scan-lookahead", "300"], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "roundtrip OK" in r.stdout and "scan: 5 boundaries" in r.stdout, (r.stdout, r.stderr[-800:])
    rows = open(out_dir / "proof.csv").read().strip().split("\n")
    assert len(rows) == 6 and rows[0].startswith("file,chunk_index,start_token,end_token,agent_text_len")
    assert [x.split(",")[1:4] for x in rows[1:]] == [[str(k), str(max(0, 512 * k - 1 - 512)), str(512 * k - 1)] for k in range(1, 6)]


@pytest.mark.parametrize("arch", ["smollm", "rwkv7"])
def test_empty_and_one_byte_files_round_trip_through_the_codec(gpu_ctx, arch):
    """Edge cases of the file-level path (src/main.rs:1979-2358 / 2485-2654): an empty file is a header plus the coder's
    finish byte 0x40 (the reference's `finish()` on an untouched encoder, src/main.rs:300-318), a one-byte file is one coded token;
    both come back byte-exact, also when more segments are asked for than there are tokens."""
    from candlezip_b200 import codec, container

    if arch == "smollm":
        model = _tiny(gpu_ctx)
    else:
        from rwkv7_weights import RWKV7_TINY, make_weights

        model = cz.Model(gpu_ctx, RWKV7_TINY)
        for name, arr in make_weights(RWKV7_TINY, 7).items():
            model.set_tensor(name, arr)
    for data, nseg in ((b"", 1), (b"", 4), (b"a", 1), (b"a", 4), (b"ab", 2)):
        blob = codec.compress(model, data, n_segments=nseg)
        f, _, _, _, _, pays = container.read_container(blob)
        assert f["token_count"] == len(data) and f["orig_len_bytes"] == len(data)
        if not data:
            assert b"".join(pays) == b"\x40"
        assert codec.decompress(model, blob) == data, (data, nseg)
