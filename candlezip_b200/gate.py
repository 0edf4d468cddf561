"""Agentic gate ("scan") over the batched hot path: SURVEY 8 a-6 / a-7, BASELINE config 4.

Mirrors the boundary block of the reference's encode loop (src/main.rs:1981-2270) without the agent subprocess: the agent
texts are an input (replayed from `agent_cache.jsonl`, src/main.rs:1152-1195, or any other source).

  reference (per boundary, sequential, on a second session)      here
  -------------------------------------------------------------  ------------------------------------------------------------
  candidates = [normalized, first 2000 bytes, digit lines,       build_candidates()
                Capitalised words]            (main.rs:2018-2032)
  budgets = [max_ctx/8, /4, /2, 3/4]          (main.rs:2034-2035)  budgets(max_ctx): 511 for SmolLM, the whole history for RWKV-7
  baseline XE + up to 16 conditioned XE passes (2043-2054)       ONE cz_xe_bits call for ALL boundaries: every (boundary,
                                                                  candidate, budget) is an independent paired stream
  best = argmax saved; gate = saved > 0 (+ thresholds) (2068-72)  same selection order (first maximum wins)
  gate: prime = tail(ids[..=i], 511 - budget) ++ hint[..budget],  cz_prime_event{i, hint, hold_until = i + lookahead,
        hold_until = i + lookahead               (2123-2149)       hist_take}: the library builds the tail itself, so the
                                                                  decoder needs only the hint tokens and the gate records
  GateRecordV2 {gate, cand, budget} -> AGT2   (main.rs:2122)      gate_records (one byte each: gate | cand<<1 | budget<<3)
"""
import numpy as np

from . import _lib

MAX_CTX_SMOLLM = 511  # max_context_length() - 1, src/models.rs:91, main.rs:2034
# RWKV-7's max_context_length() is usize::MAX (src/models.rs:150): every budget covers the whole hint, every history tail the whole
# history (BOS first), so a gated prime re-feeds everything before the boundary (models.rs:162-170)
MAX_CTX_RWKV7 = (1 << 64) - 1


def max_ctx_for(model):
    """the gate's max_ctx for a model: SmolLM's 511, or the whole history on RWKV-7"""
    return MAX_CTX_RWKV7 if model.cfg.get("arch", _lib.CZ_ARCH_SMOLLM) == _lib.CZ_ARCH_RWKV7 else MAX_CTX_SMOLLM


def build_candidates(agent_text: str):
    """src/main.rs:2018-2032 (the Rust slices the first 2000 BYTES of the normalized string)"""
    normalized = "".join(" " if (ord(c) < 32 or 127 <= ord(c) < 160) else c for c in agent_text)
    raw = normalized.encode("utf-8")
    head = raw[:2000].decode("utf-8", errors="ignore") if len(raw) > 2000 else normalized
    nums = "\n".join(l for l in normalized.split("\n") if any(c.isascii() and c.isdigit() for c in l))
    caps = " ".join(w for w in normalized.split() if w[:1].isascii() and w[:1].isupper())
    return [normalized, head, nums, caps]


def budgets(max_ctx=MAX_CTX_SMOLLM):
    return [max_ctx // 8, max_ctx // 4, max_ctx // 2, (max_ctx * 3) // 4]


def plan_scan(ids, agent_texts, tokenize_hint, agent_chunk, scan_lookahead=512, scan_max_hint_tokens=512, bos=0,
              max_ctx=MAX_CTX_SMOLLM, share_jobs=None):
    """Builds the XE jobs of every boundary.  ids: coded tokens (no BOS).  agent_texts: {chunk_index: text} (1-based chunk
    index = boundary / agent_chunk, main.rs:1985).  Returns (jobs, plan) with plan[k] = dict(i, chunk_index, job0, hints, slots)
    where jobs[job0] is the baseline and jobs[slots[cid*4 + bid]] the conditioned stream (slot None when it equals the
    baseline: empty hint, main.rs:2050).
    share_jobs: conditioned jobs of a boundary with the same prime share one stream (several slots name the same job).  The
    default shares under the whole-history rule (max_ctx = MAX_CTX_RWKV7), where the four budgets of a candidate always give the
    same prime; with SmolLM's 511 every slot keeps a stream of its own, one per XE pass of the reference."""
    seq = np.concatenate([[bos], np.asarray(ids, np.uint32)]).astype(np.uint32)  # the reference's `ids` (BOS first)
    n = len(seq) - 1
    bud = budgets(max_ctx)
    share = max_ctx == MAX_CTX_RWKV7 if share_jobs is None else bool(share_jobs)
    jobs, plan = [], []
    boundary = agent_chunk
    for i in range(n):
        if i + 1 != boundary:
            continue
        boundary += agent_chunk
        chunk_index = (i + 1) // agent_chunk
        end = min(i + scan_lookahead, len(seq))
        targets = seq[i:end]  # main.rs:2036-2038: starts AT ids[chunk_end], as the reference does
        if len(targets) == 0:
            continue
        hist = seq[max(0, i - min(max_ctx, i)):i]  # main.rs:2043-2044
        cands = build_candidates(agent_texts.get(chunk_index, ""))
        hints = [np.asarray(tokenize_hint(c, scan_max_hint_tokens), np.uint32) for c in cands]
        entry = dict(i=i, chunk_index=chunk_index, job0=len(jobs), hints=hints, slots=[])
        jobs.append((xe_prime(hist, None, max_ctx), targets))
        seen = {}  # prime bytes -> job index (same boundary, so the same targets)
        for cid in range(4):
            for bid in range(4):
                h = hints[cid][: bud[bid]]
                if len(h) == 0:
                    entry["slots"].append(None)
                    continue
                prime = xe_prime(hist, h, max_ctx)
                key = prime.tobytes()
                if not share or key not in seen:
                    seen[key] = len(jobs)
                    jobs.append((prime, targets))
                entry["slots"].append(seen[key])
        plan.append(entry)
    return jobs, plan


def xe_prime(history, hint, max_ctx=MAX_CTX_SMOLLM):
    """prime = tail(history, max_ctx - |hint|) ++ hint[..max_ctx]   (src/main.rs:1727-1739)"""
    hint = np.zeros(0, np.uint32) if hint is None else np.asarray(hint, np.uint32)
    hb = min(len(hint), max_ctx)
    take = min(max_ctx - hb, len(history))
    return np.concatenate([history[len(history) - take:], hint[:hb]]).astype(np.uint32)


def decide(plan, bits, scan_lookahead=512, thr_abs_bits=0.0, thr_pct=0.0, max_ctx=MAX_CTX_SMOLLM):
    """Selection + gate (main.rs:2046-2072) and the resulting prime events (2123-2149).  Returns (records, events, rows):
    records: one byte per boundary (gate | cand<<1 | budget<<3, main.rs:658-670); events: cz_prime_event tuples
    (i, hint tokens, hold_until, hist_take); rows: proof.csv-like dicts."""
    bud = budgets(max_ctx)
    records, events, rows = [], [], []
    for e in plan:
        base = float(bits[e["job0"]])
        best_saved, best_cond, best_cid, best_bid = -np.inf, 0.0, 0, 2
        for cid in range(4):
            for bid in range(4):
                slot = e["slots"][cid * 4 + bid]
                cond = base if slot is None else float(bits[slot])
                saved = base - cond
                if saved > best_saved:
                    best_saved, best_cond, best_cid, best_bid = saved, cond, cid, bid
        pct = best_saved / base if base > 0 else 0.0
        abs_ok = best_saved >= thr_abs_bits if thr_abs_bits > 0 else True
        pct_ok = pct * 100.0 >= thr_pct if thr_pct > 0 else True
        gate = 1 if (best_saved > 0 and abs_ok and pct_ok) else 0
        records.append(gate | (best_cid << 1) | (best_bid << 3))
        rows.append(dict(chunk_index=e["chunk_index"], i=e["i"], baseline_bits=base, conditioned_bits=best_cond, bits_saved=best_saved,
                         percent_saved=pct, gate=gate, candidate_id=best_cid, budget_id=best_bid))
        if gate:
            i, b = e["i"], bud[best_bid]
            hint = e["hints"][best_cid][:b]
            hist_take = min(max(max_ctx - b, 0), i + 1)  # history = ids[..=i] (BOS first): main.rs:2132-2134
            events.append((i, hint, i + scan_lookahead, hist_take))
    return records, events, rows


def events_from_records(records, hints_by_boundary, agent_chunk, n_tokens, scan_lookahead=512, max_ctx=MAX_CTX_SMOLLM):
    """Decode side (main.rs:2543-2614): the gate records from the container + the same agent texts give the same events.
    hints_by_boundary[k]: the four candidate hint token arrays of the k-th boundary (in boundary order)."""
    bud = budgets(max_ctx)
    events, k = [], 0
    boundary = agent_chunk
    for i in range(n_tokens):
        if i + 1 != boundary:
            continue
        boundary += agent_chunk
        if k >= len(records):
            break
        r = records[k]
        gate, cid, bid = r & 1, (r >> 1) & 3, (r >> 3) & 3
        if gate:
            b = bud[bid]
            events.append((i, np.asarray(hints_by_boundary[k][cid][:b], np.uint32), i + scan_lookahead, min(max(max_ctx - b, 0), i + 1)))
        k += 1
    return events


def scan_encode(model, ids, agent_texts, tokenize_hint, agent_chunk, n_segments=1, max_ctx=None, **kw):
    """compress with the agentic gate: one batched XE scan, then one batched encode with the gated hint primes.
    max_ctx: default max_ctx_for(model).  Returns (payloads, seg_start, records, rows, events)."""
    if n_segments != 1:
        raise ValueError("the gate works on a single AC stream (the reference's container has one)")
    max_ctx = max_ctx_for(model) if max_ctx is None else max_ctx
    look = kw.get("scan_lookahead", 512)
    jobs, plan = plan_scan(ids, agent_texts, tokenize_hint, agent_chunk, look, kw.get("scan_max_hint_tokens", 512), kw.get("bos", 0),
                           max_ctx=max_ctx)
    bits = model.xe_bits(jobs) if jobs else np.zeros(0)
    records, events, rows = decide(plan, bits, look, kw.get("thr_abs_bits", 0.0), kw.get("thr_pct", 0.0), max_ctx=max_ctx)
    pays, seg = model.encode(ids, n_segments=1, bos=kw.get("bos", 0), events=events or None)
    return pays, seg, records, rows, events


# ---------------------------------------------------------------------------------------------------------------------
# Replay of a finished run (BASELINE config 4): `--reuse-scan-dir` (src/main.rs:1966-1978) loads agent_cache.jsonl and
# proof.csv (loaders: src/main.rs:1152-1195) and never calls the agent.
# ---------------------------------------------------------------------------------------------------------------------
PROOF_HEADER = ["file", "chunk_index", "start_token", "end_token", "agent_text_len", "agent_duration_ms", "cross_entropy_baseline_bits",
                "cross_entropy_conditioned_bits", "bits_saved", "percent_saved", "agent_calls", "gate", "candidate_id", "budget_id",
                # SIMDL v1.1 columns (src/main.rs:1901-1908)
                "gate_bits", "price_transcript_bits", "price_pointer_bits", "tool_id_best", "tool_snapshot_id", "args_hash", "output_hash",
                "domain", "agent_id", "toolset_id", "run_id", "chunk_id"]


def load_replay(src):
    """src: a run directory holding agent_cache.jsonl + proof.csv (the reference's own layout), or the dict form of the
    committed fixtures (tests/golden/corpus.py::replay).  Returns (texts, calls, decisions, proof_rows):
      texts[chunk_index] = agent text, calls[chunk_index] = agent_calls        (load_cached_agent_results, main.rs:1152-1175)
      decisions[chunk_index] = (gate, candidate_id, budget_id)                   (load_gate_decisions_from_csv, main.rs:1177-1195:
                                                                                  columns 1, 11, 12, 13 of rows with >= 13 fields)
      proof_rows = the ledger rows as lists of strings (header excluded)"""
    import csv
    import io
    import json
    import os

    if isinstance(src, dict):
        cache = {int(k): v for k, v in src["agent_cache"].items()}
        rows = [list(r) for r in src["proof_rows"]]
    else:
        cache = {}
        p = os.path.join(src, "agent_cache.jsonl")
        if os.path.exists(p):
            for line in open(p, encoding="utf-8"):
                if not line.strip():
                    continue
                try:
                    v = json.loads(line)
                except ValueError:
                    continue
                if isinstance(v.get("chunk_index"), int) and isinstance(v.get("agent_text"), str) and isinstance(v.get("agent_calls"), int):
                    cache[v["chunk_index"]] = {"agent_text": v["agent_text"], "agent_calls": v["agent_calls"]}  # later lines win
        rows = []
        p = os.path.join(src, "proof.csv")
        if os.path.exists(p):
            rows = list(csv.reader(io.StringIO(open(p, encoding="utf-8", newline="").read())))[1:]
    texts = {k: v["agent_text"] for k, v in cache.items()}
    calls = {k: int(v["agent_calls"]) for k, v in cache.items()}
    decisions = {}
    for r in rows:
        if len(r) >= 13:  # the reference splits on ',' and needs parts[13]; a text-free numeric row never contains a quoted comma
            try:
                decisions[int(r[1])] = (int(r[11]), int(r[12]), int(r[13]))
            except (ValueError, IndexError):
                pass
    return texts, calls, decisions, rows


def events_from_decisions(ids, agent_texts, decisions, tokenize_hint, agent_chunk, scan_lookahead=512, scan_max_hint_tokens=512,
                          max_ctx=MAX_CTX_SMOLLM):
    """Reuse-mode encode (src/main.rs:2221-2268) and decode (2545-2614): no XE evaluation, the cached (gate, candidate, budget) of
    each boundary is applied as-is; a gated boundary without a cached agent text primes with the history tail alone.  Returns
    (records, events): AGT2 record bytes for every boundary and the cz_prime_event tuples."""
    n = len(ids)
    bud = budgets(max_ctx)
    records, events = [], []
    boundary = agent_chunk
    while boundary <= n:
        i = boundary - 1
        chunk_index = boundary // agent_chunk
        boundary += agent_chunk
        gate, cid, bid = decisions.get(chunk_index, (0, 0, 2))
        records.append((gate & 1) | ((cid & 3) << 1) | ((bid & 3) << 3))
        if gate == 1:
            cand = build_candidates(agent_texts.get(chunk_index, ""))[cid]
            hint = np.asarray(tokenize_hint(cand, scan_max_hint_tokens), np.uint32)[: bud[bid]]
            events.append((i, hint, i + scan_lookahead, min(max(max_ctx - bud[bid], 0), i + 1)))
    return records, events


def ledger_rows(rows, input_file, agent_texts, agent_calls=None, agent_chunk=512, domain="unknown", agent_id="replay", policy="aligned",
                run_id="replay", price_transcript_bits=None, doc_size_bytes=0):
    """proof.csv rows in the reference's format (src/main.rs:2177-2202): the 26 columns of PROOF_HEADER, numbers formatted
    with six decimals exactly as `format!("{:.6}")` does.  `rows` are decide()'s dicts.  price_transcript_bits(text) -> bits
    (the reference compresses the agent text with zstd level 19, main.rs:1031-1035; zstd is not in this image, so the column is 0
    unless a callable is given); the pointer price is ceil(log2(n_docs)) + ceil(log2(doc bytes)) + ceil(log2(1024)) (1038-1053)."""
    import math
    import os

    from . import container

    stem = os.path.splitext(os.path.basename(input_file))[0]
    out = []
    for r in rows:
        ci, i = r["chunk_index"], r["i"]
        text = agent_texts.get(ci, "")
        tb = text.encode("utf-8")
        h = container.blake3_16(tb).hex()
        ptr = (1 + (1 if doc_size_bytes <= 1 else math.ceil(math.log2(doc_size_bytes))) + 10) if text else 0
        out.append([input_file, str(ci), str(max(0, i - agent_chunk)), str(i), str(len(tb)), "0", f"{r['baseline_bits']:.6f}",
                    f"{r['conditioned_bits']:.6f}", f"{r['bits_saved']:.6f}", f"{r['percent_saved'] * 100.0:.6f}",
                    str((agent_calls or {}).get(ci, 0)), str(r["gate"]), str(r["candidate_id"]), str(r["budget_id"]),
                    "5" if r["gate"] else "0", str(price_transcript_bits(text) if (price_transcript_bits and text) else 0), str(ptr),
                    f"cand_{r['candidate_id']}_bud_{r['budget_id']}" if r["gate"] else "none", f"snap_{ci}", h, h, domain, agent_id,
                    f"policy_{policy}", run_id, f"{stem}:{ci}"])
    return out


def write_proof_csv(path, ledger):
    import csv

    with open(path, "w", newline="", encoding="utf-8") as f:
        w = csv.writer(f, lineterminator="\n")
        w.writerow(PROOF_HEADER)
        w.writerows(ledger)
