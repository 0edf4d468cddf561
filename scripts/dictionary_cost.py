#!/usr/bin/env python3
"""What a preset dictionary costs (GPU box only).
    python scripts/dictionary_cost.py [out.json = profiles/dictionary_r07.json]
Workload: seeded random-init models (seed 0): SmolLM-135M and RWKV-7 0.1B, byte-level ids, one segment per file.  Files are cut from the
enwik8 3 MiB stand-in; the dictionary is the first 4 KiB of alice29.txt (4,096 symbols).  Random weights do not use context, so payload
sizes are reported but say nothing about what a real dictionary saves.
  many          compress_many / decompress_many of 768 x 4 KiB files without and with the dictionary, both models; the extra time
  rwkv_naive    RWKV-7: encode of 256 x 4 KiB files under a 16,384-symbol dictionary (run once, state broadcast) against the naive
                equivalent, each file coded as D ++ T with the dictionary part dropped; model rows of each, intervals asserted equal
  smollm_decode SmolLM decompress_many without and with the dictionary at 768 streams (768 x 4 KiB) and 2,048 streams (2,048 x 1,536 B,
                all the stand-in holds); with the dictionary, a torch.profiler run of the call on the first 600 bytes of each file gives the kernel time
                of the first chunk's one-stream prime (the kernels from the decoder init to kv_prefix_broadcast_kernel) and of the broadcast
Host clock around each call (every call ends in a device synchronise); each arm is warmed up first.  The GPU's name and power limit are
read (query only) in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import codec  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "dictionary_r07.json")
res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()}
data = corpus.load("enwik8_3mib")
DIC = corpus.load("alice29.txt")[:4096]
files = [data[k * 4096 : (k + 1) * 4096] for k in range(768)]
files_2048 = [data[k * 1536 : (k + 1) * 1536] for k in range(2048)]
assert all(len(f) == 4096 for f in files) and all(len(f) == 1536 for f in files_2048)
ctx = cz.Context(0)


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def save():
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)


res["many"] = {}
for name, cfg in (("smollm_135m", cz.SMOLLM_135M), ("rwkv7_0p1b", cz.RWKV7_0P1B)):
    model = cz.Model(ctx, cfg).random_init(0, 0.02, 0.02)
    w = files[0][:600], files[1][:300]
    for d in (None, DIC):  # warm-up of both arms
        assert codec.decompress_many(model, codec.compress_many(model, list(w), dictionary=d), dictionary=d) == list(w)
    r = {}
    for label, d in (("none", None), ("dict_4k", DIC)):
        blobs, t_c = timed(lambda: codec.compress_many(model, files, dictionary=d))
        back, t_d = timed(lambda: codec.decompress_many(model, blobs, dictionary=d))
        assert back == files
        r[label] = {"compress_many_s": t_c, "decompress_many_s": t_d, "container_bytes": sum(map(len, blobs))}
    r["extra_compress_s"] = r["dict_4k"]["compress_many_s"] - r["none"]["compress_many_s"]
    r["extra_decompress_s"] = r["dict_4k"]["decompress_many_s"] - r["none"]["decompress_many_s"]
    res["many"][name] = r
    print(name, json.dumps(r), flush=True)
    save()
    model.close()

# ---- RWKV-7: state broadcast against coding D ++ T per file ----
model = cz.Model(ctx, cz.RWKV7_0P1B).random_init(0, 0.02, 0.02)
rng = np.random.default_rng(1)
D = rng.integers(0, cz.RWKV7_0P1B["vocab"], 16384).astype(np.uint32)
sub = [np.frombuffer(f, np.uint8).astype(np.uint32) for f in files[:256]]
ids = np.concatenate(sub).astype(np.uint32)
seg = np.concatenate([[0], np.cumsum([len(x) for x in sub])]).astype(np.uint64)
naive_ids = np.concatenate([np.concatenate([D, x]) for x in sub]).astype(np.uint32)
naive_seg = np.concatenate([[0], np.cumsum([len(D) + len(x) for x in sub])]).astype(np.uint64)
model.analyze(ids[:5000], seg_start=np.array([0, 2000, 5000], np.uint64), dictionary=D[:100])  # warm-up
model.analyze(naive_ids[:5000], seg_start=np.array([0, 2000, 5000], np.uint64))
r_b, t_b = timed(lambda: model.analyze(ids, seg_start=seg, dictionary=D))
r_n, t_n = timed(lambda: model.analyze(naive_ids, seg_start=naive_seg))
keep = np.concatenate([np.arange(int(naive_seg[g]) + len(D), int(naive_seg[g + 1])) for g in range(len(sub))])
equal = bool(np.array_equal(r_b["c_lo"], r_n["c_lo"][keep]) and np.array_equal(r_b["c_hi"], r_n["c_hi"][keep]))
assert equal, "broadcast intervals differ from the naive D ++ T intervals"
res["rwkv_naive"] = {"files": len(sub), "file_bytes": 4096, "dictionary_symbols": int(len(D)), "broadcast_s": t_b, "naive_s": t_n,
                     "model_rows_broadcast": int(len(D) + len(ids)), "model_rows_naive": int(len(naive_ids)),
                     "intervals_equal": equal, "speedup": t_n / t_b}
print("rwkv_naive", json.dumps(res["rwkv_naive"]), flush=True)
save()
model.close()

# ---- SmolLM decode: whole decompress_many, and the first chunk's shared prime ----
model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
res["smollm_decode"] = {}
for label, fl in (("768_streams", files), ("2048_streams", files_2048)):
    r = {"files": len(fl), "file_bytes": len(fl[0])}
    for arm, d in (("none", None), ("dict_4k", DIC)):
        blobs = codec.compress_many(model, fl, dictionary=d)
        codec.decompress_many(model, blobs[:4], dictionary=d)  # warm-up
        back, t = timed(lambda: codec.decompress_many(model, blobs, dictionary=d))
        assert back == fl
        r[arm + "_s"] = t
        if d is not None:
            try:
                from torch.profiler import ProfilerActivity, profile

                # (the first 600 bytes of every file: the same streams and the same first chunk, a trace short enough to read back)
                short = codec.compress_many(model, [f[:600] for f in fl], dictionary=d)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    codec.decompress_many(model, short, dictionary=d)
                ks = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
                i0 = next(i for i, e in enumerate(ks) if "ac_decoder_init_kernel" in e.name)
                i1 = next(i for i, e in enumerate(ks) if "kv_prefix_broadcast_kernel" in e.name)
                r["first_chunk_prefill_kernels_ms"] = sum(e.time_range.elapsed_us() for e in ks[i0 + 1 : i1]) / 1e3
                r["first_chunk_prefill_span_ms"] = (ks[i1].time_range.start - ks[i0].time_range.end) / 1e3
                r["kv_prefix_broadcast_ms"] = ks[i1].time_range.elapsed_us() / 1e3
            except Exception as e:  # the profile is an extra: the timings above stand without it
                r["profile_error"] = repr(e)
    r["extra_s"] = r["dict_4k_s"] - r["none_s"]
    res["smollm_decode"][label] = r
    print(label, json.dumps(r), flush=True)
    save()
print(f"wrote {out_path}")
