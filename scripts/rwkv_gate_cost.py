#!/usr/bin/env python3
"""What the agentic gate costs on RWKV-7, where a gated prime re-feeds the whole history (max_context_length() = usize::MAX,
src/models.rs:150; re-prime = zero state + feed, models.rs:162-170), so the work grows as n^2 / agent_chunk (GPU box only).
    python scripts/rwkv_gate_cost.py [out.json = profiles/rwkv_gate_r06.json] [--parent DIR]
Workload: RWKV-7 0.1B shape, seeded random init; the first 77 x 512 bytes of the enwik8 stand-in as spread token ids
(tests/golden/corpus.py::spread_map); the shipped asyoulik replay texts (corpus.replay("asyoulik")) as agent texts, agent_chunk 512,
lookahead 512.  Reported:
  scan      plan_scan + one cz_xe_bits call over all baseline / conditioned jobs (identical jobs shared), host clock around a
            synchronous call; its prime and target rows
  encode    gated and ungated cz_encode; the gated primes' rows
  decode    gated and ungated cz_decode (CUDA graph per unit), ms per coded token
  parent    with --parent DIR (a build of the parent commit's package, DIR/candlezip_b200): ungated decode of the same stream there and
            here, each in a worker process, alternated; launches per decode (cz_launch_count) and time
Times are host clocks around calls that end in a device synchronise.  The GPU's name and power limit are read (query only) in the
same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_TOKENS, CHUNK, LOOK = 77 * 512, 512, 512


def summary(x):
    x = np.asarray(x, np.float64)
    return {"median": float(np.median(x)), "min": float(x.min()), "max": float(x.max()),
            "spread_pct": float(100 * (x.max() - x.min()) / np.median(x)), "all": [round(float(v), 4) for v in x]}


def setup(pkg_root):
    sys.path[:0] = [pkg_root, os.path.join(ROOT, "tests", "golden")]
    import candlezip_b200 as cz
    import corpus

    ctx = cz.Context(0)
    model = cz.Model(ctx, cz.RWKV7_0P1B).random_init(0, 0.02, 0.02)
    ids = corpus.byte_ids(corpus.load("enwik8_3mib")[:N_TOKENS], cz.RWKV7_0P1B["vocab"], spread=True).astype(np.uint32)
    return cz, corpus, ctx, model, ids


def worker(pkg_root):
    """ungated decode of the workload, once per input line: prints {"s": seconds, "launches": n}"""
    cz, _, ctx, model, ids = setup(pkg_root)
    pays, seg = model.encode(ids, n_segments=1)
    for _ in sys.stdin:
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        out = model.decode(pays, seg)
        dt = time.perf_counter() - t0
        assert np.array_equal(out, ids)
        print(json.dumps({"s": dt, "launches": ctx.launch_count() - l0, "payload": len(pays[0])}), flush=True)


def main():
    args = sys.argv[1:]
    parent = None
    if "--parent" in args:
        k = args.index("--parent")
        parent = args[k + 1]
        del args[k:k + 2]
    out_path = args[0] if args else os.path.join(ROOT, "profiles", "rwkv_gate_r06.json")
    res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                 capture_output=True, text=True).stdout.strip(),
           "workload": f"RWKV-7 0.1B random init (seed 0, std 0.02); {N_TOKENS} tokens (77 x 512) of the enwik8 stand-in, spread ids; "
                       f"asyoulik replay texts; agent_chunk {CHUNK}, lookahead {LOOK}"}
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)

    def save():  # after every phase, so a run cut short keeps what it measured
        with open(out_path, "w") as f:
            json.dump(res, f, indent=1)

    cz, corpus, ctx, model, ids = setup(ROOT)
    from candlezip_b200 import gate

    V = cz.RWKV7_0P1B["vocab"]
    texts, _, _, _ = gate.load_replay(corpus.replay("asyoulik"))
    m = corpus.spread_map(V)
    tok = lambda text, mx: m[np.frombuffer(text.encode("utf-8"), np.uint8)][:mx]  # noqa: E731
    big = gate.max_ctx_for(model)
    # ---- scan ----
    scan_s = []
    for _ in range(3):  # the first call is the warm-up
        t0 = time.perf_counter()
        jobs, plan = gate.plan_scan(ids, texts, tok, CHUNK, LOOK, max_ctx=big)
        bits = model.xe_bits(jobs)
        scan_s.append(time.perf_counter() - t0)
    unshared = gate.plan_scan(ids, texts, tok, CHUNK, LOOK, max_ctx=big, share_jobs=False)[0]
    records, events, rows = gate.decide(plan, bits, LOOK, max_ctx=big)
    res["scan"] = {"boundaries": len(plan), "jobs": len(jobs), "jobs_without_sharing": len(unshared),
                   "prime_rows": int(sum(len(p) for p, _ in jobs)), "target_rows": int(sum(len(t) for _, t in jobs)),
                   "prime_rows_without_sharing": int(sum(len(p) for p, _ in unshared)), "seconds": summary(scan_s[1:])}
    print("scan", json.dumps(res["scan"]), flush=True)
    save()
    # ---- encode ----
    gated_rows = int(sum(min(ht, i + 1) + len(h) for i, h, _, ht in events))  # byte-spread ids: no literal escapes, BOS pads
    enc = {"gated": [], "ungated": []}
    for _ in range(3):
        for name, ev in (("gated", events), ("ungated", None)):
            t0 = time.perf_counter()
            pays, seg = model.encode(ids, n_segments=1, events=ev)
            enc[name].append(time.perf_counter() - t0)
            if name == "gated":
                gp = pays
            else:
                up = pays
    res["encode"] = {"events": len(events), "prime_rows": gated_rows, "payload_bytes_gated": len(gp[0]), "payload_bytes_ungated": len(up[0]),
                     "seconds_gated": summary(enc["gated"][1:]), "seconds_ungated": summary(enc["ungated"][1:])}
    print("encode", json.dumps(res["encode"]), flush=True)
    save()
    # ---- decode ----
    dec = {"gated": [], "ungated": []}
    launches = {}
    for _ in range(2):  # (modules and buffers are warm from the encode calls)
        for name, pays, ev in (("gated", gp, events), ("ungated", up, None)):
            l0 = ctx.launch_count()
            t0 = time.perf_counter()
            out = model.decode(pays, seg, events=ev)
            dec[name].append(time.perf_counter() - t0)
            launches[name] = ctx.launch_count() - l0
            assert np.array_equal(out, ids), name
            print("decode", name, round(dec[name][-1], 3), flush=True)
    res["decode"] = {name: {"seconds": summary(v), "ms_per_token": summary(np.asarray(v) * 1e3 / N_TOKENS), "launches": launches[name]}
                     for name, v in dec.items()}
    save()
    # ---- ungated decode against the parent commit ----
    if parent:
        ws = {name: subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", root], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                     text=True, cwd=ROOT)
              for name, root in (("this", ROOT), ("parent", os.path.abspath(parent)))}
        got = {name: [] for name in ws}
        try:
            for rep in range(3):  # the first round is the warm-up
                for name, w in ws.items():
                    w.stdin.write("go\n")
                    w.stdin.flush()
                    r = json.loads(w.stdout.readline())
                    print("ungated decode", name, rep, r, flush=True)
                    if rep:
                        got[name].append(r)
        finally:
            for w in ws.values():
                w.stdin.close()
                w.wait(timeout=600)
        res["ungated_decode_vs_parent"] = {name: {"seconds": summary([r["s"] for r in v]), "launches": sorted({r["launches"] for r in v}),
                                                  "payload_bytes": sorted({r["payload"] for r in v})} for name, v in got.items()}
    else:
        res["ungated_decode_vs_parent"] = "not measured"
    save()
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--worker":
        worker(sys.argv[2])
    else:
        main()
