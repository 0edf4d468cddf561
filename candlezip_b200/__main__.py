"""`python -m candlezip_b200 {compress,decompress,self-test}`: a thin twin of the reference CLI's hot-path surface
(src/main.rs:34-221: compress | decompress | self-test, --backend smollm|rwkv7, --context, --reprime-interval) over the
batched B200 path.  Out of scope here, as in DESIGN.md: hf-hub download, agents, watchdog logging.

Weights: --weights *.safetensors (HF LLaMA / candle_rwkv7 tensor names) or --random-init SEED (no checkpoints exist offline).
Tokenizer: --tokenizer tokenizer.json (HF `tokenizers`, SmolLM) or a RWKV vocab json; default = byte-level ids (lossless for
every input).  --segments N > 1 writes the SEG1 container extension (parallel decode); N = 1 is the reference's v2 layout.
--on-zero-width {stored,floor}: what compress does when the SmolLM coder meets a token of mass < 2^-30 (codec.compress).
compress-many / decompress-many IN... [--out-dir DIR]: many files through one encode call and lock-step decode waves of at most
--max-streams streams (codec.compress_many / decompress_many); each .canz is the one `compress` writes for that file.
analyze INPUT [OUTPUT]: per-token code lengths, coding-distribution entropies and positions (codec.analyze), tokenised and split as
`compress` does, into OUTPUT (default INPUT.analysis.npz: the arrays, plus the summary as JSON under "summary"); prints the summary.
--pdf-floor (analyze, SmolLM only) codes with the floored pdf.
--dictionary FILE (every command but the gate replay): code each segment as if it followed FILE's contents (a preset dictionary, never
stored in the container); decompress needs the same FILE.
--match-order K (compress, self-test, compress-many; not with the gate replay or analyze): code with the match model of order K (1..16),
which predicts a token that repeats an earlier context of its segment; the container records K.
"""
import argparse
import json
import sys
import time

import numpy as np

from . import RWKV7_0P1B, SMOLLM_135M, Context, Model, codec, container, gate


class HfTokenizer:
    """tok.encode(from_utf8_lossy(data), add_special_tokens=false) / tok.decode(ids, skip_special_tokens=true): the reference's
    SmolLM tokenisation (src/main.rs:1850-1857, 2654).  Lossy for non-UTF-8 input exactly like the reference; decompress()
    verifies the BLAKE3 of the decoded bytes and reports a mismatch instead of silently returning different bytes."""

    def __init__(self, path):
        from tokenizers import Tokenizer

        self.tok = Tokenizer.from_file(path)

    def encode_bytes(self, data: bytes):
        return np.asarray(self.tok.encode(data.decode("utf-8", errors="replace"), add_special_tokens=False).ids, np.uint32)

    def decode_bytes(self, ids):
        return self.tok.decode([int(t) for t in ids], skip_special_tokens=True).encode("utf-8")


def _model(args):
    ctx = Context(args.device)
    cfg = SMOLLM_135M if args.backend == "smollm" else RWKV7_0P1B
    m = Model(ctx, cfg)
    if args.weights:
        m.load_safetensors(args.weights)
    else:
        m.random_init(args.random_init, 0.02, 0.02)
    tok = None
    if args.tokenizer:
        tok = HfTokenizer(args.tokenizer) if args.backend == "smollm" else codec.RwkvTokenizer.from_json(args.tokenizer)
    return m, tok


def _hint_tokenizer(tok, vocab):
    """tokenize_hint_smol (src/main.rs:1712-1717): encode the candidate text, keep at most max_tokens ids"""
    if tok is None:  # byte-level ids offline
        return lambda text, mx: np.frombuffer(text.encode("utf-8"), np.uint8).astype(np.uint32)[:mx]
    return lambda text, mx: tok.encode_bytes(text.encode("utf-8"))[:mx]


def _scan_compress(model, tok, data, args):
    """`--reuse-scan-dir DIR` (src/main.rs:1966-1978): the agentic gate replayed from DIR/agent_cache.jsonl (+ proof.csv), no agent
    process.  The baseline / hint-conditioned cross-entropy passes of every boundary run as one batch of paired streams; gated hints
    prime the main stream; the container carries the AGT2 records; a proof.csv in the reference's format goes to --scan-output-dir."""
    import os

    ids = codec.tokenize(model, data, tok or codec.ByteTokenizer())  # RWKV-7: literal escapes for what the vocabulary cannot cover
    texts, calls, decisions, _ = gate.load_replay(args.reuse_scan_dir)
    hint_tok = _hint_tokenizer(tok, model.cfg["vocab"])
    pays, seg, records, rows, events = gate.scan_encode(model, ids, texts, hint_tok, agent_chunk=args.agent_chunk,
                                                        scan_lookahead=args.scan_lookahead, thr_abs_bits=args.scan_gate_threshold_abs_bits,
                                                        thr_pct=args.scan_gate_threshold_pct)
    flags = int(container.lib.cz_flags_pack(1, 0, 1, args.agent_chunk))
    fields = dict(token_count=len(ids), orig_len_bytes=len(data), vocab_size=int(model.cfg["vocab"]), context_window=args.context,
                  reprime_interval=args.reprime_interval, orig_hash16=container.blake3_16(data), reserved_flags=flags)
    blob = container.write_container(fields, b"model.safetensors", pays, gates=records)
    if args.scan_output_dir:
        os.makedirs(args.scan_output_dir, exist_ok=True)
        gate.write_proof_csv(os.path.join(args.scan_output_dir, "proof.csv"),
                             gate.ledger_rows(rows, args.input, texts, calls, agent_chunk=args.agent_chunk, doc_size_bytes=len(data)))
    saved = sum(max(r["bits_saved"], 0.0) for r in rows)
    print(f"scan: {len(rows)} boundaries, {sum(r['gate'] for r in rows)} gated, {saved:.1f} bits saved over the scanned spans")
    return blob


def _scan_decompress(model, tok, blob, args):
    """decode side of the gate (src/main.rs:2543-2614): AGT2 records from the container + the same agent texts rebuild the primes"""
    f, _, records, _, _, pays = container.read_container(blob)
    n = int(f["token_count"])
    chunk = int(f["reserved_flags"]) >> 16
    texts, _, _, _ = gate.load_replay(args.reuse_scan_dir)
    hint_tok = _hint_tokenizer(tok, model.cfg["vocab"])
    hints = [[np.asarray(hint_tok(c, 512), np.uint32) for c in gate.build_candidates(texts.get(k + 1, ""))] for k in range(len(records or []))]
    events = gate.events_from_records(records or [], hints, chunk, n, scan_lookahead=args.scan_lookahead, max_ctx=gate.max_ctx_for(model))
    ids = model.decode(pays, np.array([0, n], np.uint64), bos=int(f["bos_token_id"]), context=int(f["context_window"]),
                       reprime_interval=int(f["reprime_interval"]), events=events or None)
    return codec._finish(model, tok or codec.ByteTokenizer(), f, ids, verify=True)


def _main_many(args, ap):
    """compress-many / decompress-many: every input in one codec.compress_many / decompress_many call"""
    import os

    ext = ".canz" if args.command == "compress-many" else ".out"
    outs = [os.path.join(args.out_dir or os.path.dirname(p), os.path.basename(p) + ext) for p in args.input]
    if len(set(map(os.path.abspath, outs))) != len(outs):
        ap.error("two inputs would write the same output file")
    model, tok = _model(args)
    datas = [open(p, "rb").read() for p in args.input]
    t0 = time.perf_counter()
    if args.command == "compress-many":
        res = codec.compress_many(model, datas, tok, args.segments, context=args.context, reprime_interval=args.reprime_interval,
                                  on_zero_width=args.on_zero_width or "stored", dictionary=args.dictionary_bytes, match_order=args.match_order)
    else:
        res = codec.decompress_many(model, datas, tok, max_streams=args.max_streams, dictionary=args.dictionary_bytes)
    dt = time.perf_counter() - t0
    if args.out_dir:
        os.makedirs(args.out_dir, exist_ok=True)
    for path, blob in zip(outs, res):
        open(path, "wb").write(blob)
    n_in, n_out = sum(map(len, datas)), sum(map(len, res))
    print(f"{len(datas)} files: {n_in} -> {n_out} bytes in {dt:.3f} s")
    return 0


def _print_summary(s):
    bpb = lambda x: "n/a" if x is None else f"{x:.4f}"  # noqa: E731
    print(f"{s['tokens']} tokens, {s['bytes']} bytes: {s['bits']:.1f} bits of code length ({bpb(s['bits_per_byte'])} bits/byte), "
          f"{s['payload_bits']} payload bits ({bpb(s['payload_bits_per_byte'])} bits/byte)")
    print(f"mean code length {s['mean_bits'] if s['mean_bits'] is None else round(s['mean_bits'], 4)} bits/token, "
          f"mean entropy {s['mean_entropy'] if s['mean_entropy'] is None else round(s['mean_entropy'], 4)} bits/token, "
          f"{s['zero_width']} zero-width tokens" + (f" (first: {s['first_zero_width']})" if s["zero_width"] else ""))
    for g, seg in enumerate(s["segments"]):
        print(f"  segment {g}: {seg['tokens']} tokens, {seg['bits']:.1f} bits, {seg['payload_bits']} payload bits")
    for name, key in (("position in chunk", "by_chunk_position"), ("position in segment", "by_segment_position")):
        print(f"  by {name}: " + ", ".join(f"{b['bucket']}: {'-' if b['mean_bits'] is None else format(b['mean_bits'], '.3f')}"
                                          f"/{b['mean_entropy']:.3f}" for b in s[key]) + "  (mean bits / mean entropy)")


def _analyze(args):
    model, tok = _model(args)
    data = open(args.input, "rb").read()
    arrays, summary = codec.analyze(model, data, tok, args.segments, context=args.context, reprime_interval=args.reprime_interval,
                                    pdf_floor=args.pdf_floor, dictionary=args.dictionary_bytes)
    out = args.output or args.input + ".analysis.npz"
    with open(out, "wb") as f:  # (a file object: np.savez would append .npz to a name without it)
        np.savez(f, summary=np.array(json.dumps(summary)), **arrays)
    _print_summary(summary)
    print(f"wrote {out}")
    return 0


def main(argv=None):
    ap = argparse.ArgumentParser(prog="candlezip_b200")
    ap.add_argument("command", choices=["compress", "decompress", "self-test", "compress-many", "decompress-many", "analyze"])
    ap.add_argument("input", nargs="+", help="INPUT [OUTPUT]; compress-many / decompress-many: one or more inputs")
    ap.add_argument("--backend", choices=["smollm", "rwkv7"], default="smollm")
    ap.add_argument("--context", type=int, default=512)
    ap.add_argument("--reprime-interval", type=int, default=512)
    ap.add_argument("--segments", type=int, help="independently coded segments per file (compress / self-test / compress-many); default 1")
    ap.add_argument("--weights", nargs="*")
    ap.add_argument("--random-init", type=int, default=0)
    ap.add_argument("--tokenizer")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--on-zero-width", choices=["stored", "floor"],
                    help="compress / self-test: a token the SmolLM coder cannot code stores the input uncoded (stored) or codes it "
                         "again with the floored pdf (floor); default stored")
    # the agentic gate, replay only (src/main.rs:74-118: --scan, --scan-lookahead, --reuse-scan-dir, gate thresholds); both backends
    ap.add_argument("--reuse-scan-dir", help="directory with agent_cache.jsonl (+ proof.csv) of a finished run: replay the gate scan")
    ap.add_argument("--scan-lookahead", type=int, default=512)
    ap.add_argument("--agent-chunk", type=int, default=512, help="tokens between gate boundaries (the reference's --scan-chunk-size in tokens)")
    ap.add_argument("--scan-gate-threshold-abs-bits", type=float, default=0.0)
    ap.add_argument("--scan-gate-threshold-pct", type=float, default=0.0)
    ap.add_argument("--scan-output-dir", help="where the proof.csv ledger of a scan goes")
    ap.add_argument("--out-dir", help="compress-many / decompress-many: where NAME.canz / NAME.out go (default: beside each input)")
    ap.add_argument("--max-streams", type=int, help="decompress-many: most segments decoded together in one lock-step wave; default 2048")
    ap.add_argument("--pdf-floor", action="store_true", help="analyze: code with the floored SmolLM pdf (no token is zero-width)")
    ap.add_argument("--dictionary", metavar="FILE", help="preset dictionary: code every segment as if it followed FILE's contents; "
                                                         "decompressing needs the same FILE")
    ap.add_argument("--match-order", type=int, metavar="K", help="compress / self-test / compress-many: code with the match model of order "
                                                                   "K (1..16); the container records it")
    args = ap.parse_args(argv)
    if args.dictionary and args.reuse_scan_dir:
        ap.error("--dictionary is not available with --reuse-scan-dir (gated hint primes and a dictionary do not combine)")
    # flags that only one side uses are refused on the other instead of being ignored
    if args.command == "decompress-many" and (args.segments is not None or args.on_zero_width):
        ap.error("--segments and --on-zero-width are compress settings: a container carries its own (decompress-many)")
    if args.command != "decompress-many" and args.max_streams is not None:
        ap.error("--max-streams applies to decompress-many only")
    if args.match_order is not None:
        if args.command not in ("compress", "self-test", "compress-many"):
            ap.error(f"--match-order is a compress setting (compress, self-test, compress-many), not available with {args.command}")
        if args.reuse_scan_dir:
            ap.error("--match-order is not available with --reuse-scan-dir (gated hint primes and the match model do not combine)")
        if not 1 <= args.match_order <= 16:
            ap.error("--match-order must be in [1, 16]")
    args.match_order = args.match_order or 0
    if args.pdf_floor and (args.command != "analyze" or args.backend != "smollm"):
        ap.error("--pdf-floor applies to analyze on the SmolLM backend only (RWKV-7 codes with a floored alphabet already)")
    if args.command == "analyze":
        for flag, val in (("--reuse-scan-dir", args.reuse_scan_dir), ("--on-zero-width", args.on_zero_width), ("--out-dir", args.out_dir),
                          ("--max-streams", args.max_streams)):
            if val is not None:
                ap.error(f"{flag} is not available with analyze")
    if args.segments is None:
        args.segments = 1
    args.dictionary_bytes = None
    if args.dictionary:
        with open(args.dictionary, "rb") as f:
            args.dictionary_bytes = f.read()
    if args.command.endswith("-many"):
        if args.reuse_scan_dir:
            ap.error("--reuse-scan-dir codes one file at a time: not available with compress-many / decompress-many")
        if args.max_streams is None:
            args.max_streams = 2048
        if args.max_streams < 1:
            ap.error("--max-streams must be >= 1")
        return _main_many(args, ap)
    if len(args.input) > 2:
        ap.error(f"{args.command} takes INPUT [OUTPUT]")
    args.input, args.output = args.input[0], (args.input[1] if len(args.input) > 1 else None)
    if args.command == "analyze":
        return _analyze(args)
    scan = bool(args.reuse_scan_dir)
    if scan and args.segments != 1:
        ap.error("--reuse-scan-dir works on one AC stream (--segments 1), like the reference's container")
    if scan and args.on_zero_width:
        ap.error("--on-zero-width is not available with --reuse-scan-dir (the gated stream has no fallback of either kind)")
    model, tok = _model(args)
    data = open(args.input, "rb").read()
    if args.command == "compress":
        blob = _scan_compress(model, tok, data, args) if scan else \
            codec.compress(model, data, tok, args.segments, context=args.context, reprime_interval=args.reprime_interval,
                           on_zero_width=args.on_zero_width or "stored", dictionary=args.dictionary_bytes, match_order=args.match_order)
        open(args.output or args.input + ".canz", "wb").write(blob)
        print(f"{len(data)} -> {len(blob)} bytes ({8 * len(blob) / max(1, len(data)):.4f} bits/byte)")
    elif args.command == "decompress":
        out = _scan_decompress(model, tok, data, args) if scan else codec.decompress(model, data, tok, dictionary=args.dictionary_bytes)
        open(args.output or args.input + ".out", "wb").write(out)
        print(f"{len(data)} -> {len(out)} bytes")
    else:  # self-test: encode + decode round trip with timings (src/main.rs:156-221)
        t0 = time.perf_counter()
        blob = _scan_compress(model, tok, data, args) if scan else \
            codec.compress(model, data, tok, args.segments, context=args.context, reprime_interval=args.reprime_interval,
                           on_zero_width=args.on_zero_width or "stored", dictionary=args.dictionary_bytes, match_order=args.match_order)
        t1 = time.perf_counter()
        out = _scan_decompress(model, tok, blob, args) if scan else codec.decompress(model, blob, tok, dictionary=args.dictionary_bytes)
        t2 = time.perf_counter()
        ok = out == data
        print(f"Compression: {t1 - t0:.3f} s  Decompression: {t2 - t1:.3f} s  {8 * len(blob) / max(1, len(data)):.4f} bits/byte  "
              f"roundtrip {'OK' if ok else 'MISMATCH'}")
        return 0 if ok else 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
