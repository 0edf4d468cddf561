#!/usr/bin/env python3
"""What the match model costs and gives (GPU box only).
    python scripts/match_cost.py [out.json = profiles/match_r08.json]
Workload: seeded random-init SmolLM-135M (seed 0), byte-level ids, K = 4.
  encode_step   bench.py's headline step: cz_encode_dev over 262,144 ids of the enwik8 stand-in (spread over the vocabulary) in 32
                segments, match off and on alternated, each warmed; CUDA events around each step; median and spread per arm, and the
                payload bytes of each arm
  many          compress_many / decompress_many of 768 x 4 KiB files of the stand-in, off and on (host clock; calls synchronise)
  decode_step   decompress_many ms per lock-step step at 768 streams (768 x 4 KiB) and 2,048 streams (2,048 x 1,536 B), off and on
  sizes         container bytes of the fixtures (one segment, encode only), off and on
The GPU's name and power limit are read (query only) in the same run."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import _lib, codec  # noqa: E402

K = 4
out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "match_r08.json")
res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip(), "match_order": K}
data = corpus.load("enwik8_3mib")
ctx = cz.Context(0)
model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)


def save():
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


# ---- bench's encode step, off / on alternated ----
import torch  # noqa: E402

n, n_seg = 262144, 32
ids_np = corpus.byte_ids(data[:n], cz.SMOLLM_135M["vocab"], spread=True).astype(np.uint32)
seg_start = cz.split_segments(n, n_seg)
sched, keep = model._schedule(n, seg_start, 0, 512, 512, None, 0)
cap = 8 * n + 8 * n_seg + 16
ids_dev = torch.from_numpy(ids_np.view(np.int32)).cuda()
out_dev = torch.empty(cap, dtype=torch.uint8, device="cuda")
seg_off = np.zeros(n_seg + 1, np.uint64)
stream = torch.cuda.ExternalStream(ctx.stream_ptr())


def step(order):
    model.set_match(order)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    _lib.check(_lib.lib.cz_encode_dev(model._h, C.c_void_p(ids_dev.data_ptr()), n, C.byref(sched), C.c_void_p(out_dev.data_ptr()), cap,
                                      seg_off.ctypes.data_as(_lib.u64p)))
    ev1.record(stream)
    ev1.synchronize()
    return ev0.elapsed_time(ev1), int(seg_off[-1])


for _ in range(3):
    step(0), step(K)
ms = {0: [], K: []}
pay = {}
for _ in range(10):
    for order in (0, K):
        t, b = step(order)
        ms[order].append(t)
        pay[order] = b
res["encode_step"] = {f"order_{o}": {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "payload_bytes": pay[o]}
                      for o, v in ms.items()}
res["encode_step"]["extra_ms_median"] = statistics.median(ms[K]) - statistics.median(ms[0])
model.set_match(0)
print("encode_step", json.dumps(res["encode_step"]), flush=True)
save()

# ---- many files, and the decode step at 768 and 2,048 streams ----
files = [data[k * 4096:(k + 1) * 4096] for k in range(768)]
files_2048 = [data[k * 1536:(k + 1) * 1536] for k in range(2048)]
w = [files[0][:600], files[1][:300]]
for o in (0, K):  # warm-up of both arms
    assert codec.decompress_many(model, codec.compress_many(model, w, match_order=o)) == w
res["many"], res["decode_step"] = {}, {}
for label, fs, steps in (("768x4KiB", files, 4096), ("2048x1536B", files_2048, 1536)):
    r = {}
    for o in (0, K):
        blobs, t_c = timed(lambda: codec.compress_many(model, fs, match_order=o))
        back, t_d = timed(lambda: codec.decompress_many(model, blobs))
        assert back == fs
        r[f"order_{o}"] = {"compress_many_s": t_c, "decompress_many_s": t_d, "decode_ms_per_step": 1e3 * t_d / steps,
                           "container_bytes": sum(map(len, blobs))}
    (res["many"] if label == "768x4KiB" else res["decode_step"])[label] = r
    if label == "768x4KiB":
        res["decode_step"][label] = {k: v["decode_ms_per_step"] for k, v in r.items()}
    print(label, json.dumps(r), flush=True)
    save()

# ---- container sizes of the fixtures ----
res["sizes"] = {}
for name, d in (("alphabet.txt", corpus.load("alphabet.txt")), ("alice29.txt", corpus.load("alice29.txt")),
                ("enwik8_first_1MiB", data[:1 << 20]), ("random_1MiB", corpus.high_entropy_stream(1 << 20))):
    r = {"bytes": len(d)}
    for o in (0, K):
        r[f"order_{o}"] = len(codec.compress(model, d, match_order=o))
    r["ratio_on_off"] = r[f"order_{K}"] / r["order_0"]
    res["sizes"][name] = r
    print(name, json.dumps(r), flush=True)
    save()
model.close()
ctx.close()
