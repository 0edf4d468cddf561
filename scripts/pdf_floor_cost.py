#!/usr/bin/env python3
"""What coding with the floored SmolLM pdf (CZ_CDF_SMOLLM_FLOOR, cz_model_set_pdf_floor) costs against the unfloored one (GPU box only).
    python scripts/pdf_floor_cost.py [out.json = profiles/pdf_floor_r03.json] [steps = 6]
The floor adds one in-order f64 pass over the vocabulary to the encode-side stats kernel and to the decode-side search.
  encode   bench.py's headline step: SmolLM-135M seeded random init, the enwik8 stand-in's first 262,144 bytes as spread token ids
           (tests/golden/corpus.py::spread_map), 32 segments, cz_encode_dev; CUDA events around each step, profiling off, the two
           modes alternated step by step after a warm-up of both
  split    a separate pass with deferred per-launch events (Context.profile(2)): the CDF full passes / decode search (`cdf`) and
           the encode-side prefix walk (`cdf_prefix`)
  decode   the lock-step decoder at 512 streams x 2,048 tokens (the first 1 MiB of the stand-in), host clock around cz_decode
  sizes    payload bytes of both modes; a peaky model (random tokens are zero-width unfloored) where the unfloored coder falls back to
           a STORED container: its size against the PDF_FLOOR container's
The GPU's name and power limit are read (query only) in the same run."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import _lib, codec, container  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "pdf_floor_r03.json")
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 6
V = 49152
res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip(), "torch_device": torch.cuda.get_device_name(0)}
ctx = cz.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream_ptr())
model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
data = corpus.load("enwik8_3mib")

# ---- encode: the headline step, both modes alternated ----
n, S = 262144, 32
ids = corpus.byte_ids(data[:n], V, True)
seg_start = cz.split_segments(n, S)
sched, keep = model._schedule(n, seg_start, 0, 512, 512, None, 0)
cap = 4 * n + 8 * S + 16
ids_dev = torch.from_numpy(ids.astype(np.int64)).to(torch.int32).cuda()
out_dev = torch.empty(cap, dtype=torch.uint8, device="cuda")
seg_off = np.zeros(S + 1, np.uint64)


def step(floor):
    _lib.check(_lib.lib.cz_model_set_pdf_floor(model._h, floor))
    _lib.check(_lib.lib.cz_encode_dev(model._h, C.c_void_p(ids_dev.data_ptr()), n, C.byref(sched), C.c_void_p(out_dev.data_ptr()), cap,
                                      seg_off.ctypes.data_as(_lib.u64p)))
    return int(seg_off[S])


payload = {}
for floor in (0, 1, 0, 1):  # warm-up of both modes (grow-only buffers, module loads)
    payload[floor] = step(floor)
ms = {0: [], 1: []}
for _ in range(steps):
    for floor in (0, 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        assert step(floor) == payload[floor]
        e1.record(stream)
        e1.synchronize()
        ms[floor].append(e0.elapsed_time(e1))


def summary(x):
    x = np.asarray(x)
    return {"median": float(np.median(x)), "min": float(x.min()), "max": float(x.max()), "spread_pct": float(100 * (x.max() - x.min()) / np.median(x)),
            "all": [round(float(v), 3) for v in x]}


res["encode"] = {"workload": f"{n} tokens (enwik8 stand-in, spread byte ids) as {S} segments per step, cz_encode_dev, SmolLM-135M random init",
                 "ms_per_step": {"mode0": summary(ms[0]), "mode2": summary(ms[1])},
                 "mode2_over_mode0": float(np.median(ms[1]) / np.median(ms[0])),
                 "payload_bytes": {"mode0": payload[0], "mode2": payload[1]}}

# ---- per-family split, a separate pass ----
split = {}
for floor in (0, 1):
    ctx.profile(2)
    ctx.profile_read(reset=True)
    for _ in range(2):
        step(floor)
    torch.cuda.synchronize()
    fam = ctx.profile_read(reset=True)
    ctx.profile(0)
    split[f"mode{2 * floor}"] = {k: round(fam[k][0] / 2, 3) for k in ("cdf", "cdf_prefix", "gemm", "attn", "coder")}
res["encode_family_ms_per_step"] = split

# ---- decode: 512 streams x 2,048 tokens ----
nd, Sd = 512 * 2048, 512
dids = corpus.byte_ids(data[:nd], V, True)
dec = {}
for floor in (False, True):
    pays, seg = model.encode(dids, n_segments=Sd, pdf_floor=floor)
    t = []
    for _ in range(2):
        t0 = time.perf_counter()
        out = model.decode(pays, seg, pdf_floor=floor)
        t.append(time.perf_counter() - t0)
        assert np.array_equal(out, dids)
    dec[f"mode{2 * int(floor)}"] = {"s": [round(x, 3) for x in t], "ms_per_step": round(1e3 * min(t) / 2048, 4), "payload_bytes": sum(map(len, pays))}
res["decode"] = {"workload": f"{Sd} streams x {nd // Sd} tokens, lock-step decoder (cz_decode), best of 2", **dec}
model.close()

# ---- a peaky model: STORED (unfloored fallback) against PDF_FLOOR ----
peaky = cz.Model(ctx, cz.SMOLLM_135M).random_init(5, 0.05, 1.5)


class SpreadTokenizer:
    def encode_bytes(self, b):
        return corpus.byte_ids(b, V, True)

    def decode_bytes(self, ids):
        return corpus.ids_to_bytes(ids, V, True)


pdata = data[:65536]
stored = codec.compress(peaky, pdata, SpreadTokenizer(), 8)
floored = codec.compress(peaky, pdata, SpreadTokenizer(), 8, on_zero_width="floor")
assert codec.decompress(peaky, floored, SpreadTokenizer()) == pdata
res["peaky_container_bytes"] = {"input": len(pdata), "model": "SmolLM-135M shape, random_init(5, 0.05, 1.5)", "segments": 8,
                                "stored_flag": bool(container.read_container(stored)[0]["reserved_flags"] & _lib.CZ_FLAG_STORED),
                                "stored": len(stored), "pdf_floor": len(floored),
                                "pdf_floor_flag": bool(container.read_container(floored)[0]["reserved_flags"] & _lib.CZ_FLAG_PDF_FLOOR)}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
json.dump(res, open(out_path, "w"), indent=1)
print(json.dumps(res, indent=1))
