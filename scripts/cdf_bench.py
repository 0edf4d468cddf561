#!/usr/bin/env python3
"""Micro-benchmark of the encode-side CDF kernels on a device-resident logits batch (GPU box only).
    python scripts/cdf_bench.py [mode=0] [cols=131072]
Times cz_cdf_bounds_dev with CUDA events for: coded symbol 0 everywhere (the full passes alone), symbols distributed like the
bench's spread byte ids, and uniform symbols; with the e-cache (`tma`) and without it (`tma_noecache`: the prefix walk reads the
logits).  The batch's row stride is `cols`.  The TMA-staged stats kernel needs a stride that is a multiple of 4, so an odd `cols`
(e.g. 131071) times the direct-load stats kernel instead, and without an e-cache in both variants."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import _lib  # noqa: E402

mode = int(sys.argv[1]) if len(sys.argv) > 1 else 0
M = int(sys.argv[2]) if len(sys.argv) > 2 else 131072
V = 65536 if mode else 49152
ctx = cz.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream_ptr())
g = torch.Generator(device="cuda").manual_seed(0)
logits0 = torch.empty((V, M), dtype=torch.float32, device="cuda")
for r in range(0, V, 4096):
    logits0[r:r + 4096].normal_(0, 1.2, generator=g)
logits = torch.empty_like(logits0)
lo = torch.empty(M, dtype=torch.int32, device="cuda")
hi = torch.empty(M, dtype=torch.int32, device="cuda")
data = corpus.load("enwik8_3mib")
ids = corpus.byte_ids((data * (M // len(data) + 1))[:M], V, True)
cases = {"sym0": np.zeros(M, np.uint32), "spread_ids": ids, "uniform": np.random.default_rng(0).integers(0, V, M).astype(np.uint32)}
res = {"mode": mode, "V": V, "cols": M}
variants = ("tma", "tma_noecache")
if os.environ.get("CDF_BENCH_VARIANTS"):
    variants = tuple(os.environ["CDF_BENCH_VARIANTS"].split(","))
for variant in variants:
    os.environ.pop("CZ_CDF_NO_ECACHE", None)
    if variant == "tma_noecache":  # the prefix walk reads the vocab-major logits instead of the e-cache the stats pass fills
        os.environ["CZ_CDF_NO_ECACHE"] = "1"
    for name, syms in cases.items():
        s_dev = torch.from_numpy(syms.astype(np.int64)).to(torch.int32).cuda()
        ts = []
        for rep in range(3):
            logits.copy_(logits0)  # (the RWKV alphabet's pass rewrites the batch in place)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            _lib.check(_lib.lib.cz_cdf_bounds_dev(ctx._h, C.c_void_p(logits.data_ptr()), V, M, M, mode, C.c_void_p(s_dev.data_ptr()),
                                                  C.c_void_p(lo.data_ptr()), C.c_void_p(hi.data_ptr())))
            e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        res[f"{variant}_{name}_ms"] = round(min(ts), 3)
        res[f"{variant}_{name}_GBps_algorithmic"] = round(4.0 * V * M * (1 + syms.astype(np.float64).mean() / V) / min(ts) / 1e6, 1)
print(json.dumps(res))
