#!/usr/bin/env python3
"""Many small files through the batch calls against one call per file (GPU box only).
    python scripts/batch_cost.py [out.json = profiles/batch_r04.json] [n_single_decode = 4]
Workload: SmolLM-135M seeded random init (seed 0), the enwik8 3 MiB stand-in cut into 768 files of 4 KiB, byte-level ids, one segment
per file (the CLI's default --segments 1, the reference's v2 layout).
  compress    codec.compress_many over all 768 files against a loop of codec.compress over the same files; the containers of both
              arms must be identical
  decompress  codec.decompress_many over all 768 containers (one lock-step wave: 768 streams) against a loop of codec.decompress over
              the first n_single_decode files (each one a single stream, one full forward per token: all 768 would take hours)
Host clock around each arm (every call ends in a device synchronise); both arms are warmed up on a short file first.
The GPU's name and power limit are read (query only) in the same run."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import codec  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "batch_r04.json")
n_single = int(sys.argv[2]) if len(sys.argv) > 2 else 4
FILE, N_FILES = 4096, 768
res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()}
ctx = cz.Context(0)
model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
data = corpus.load("enwik8_3mib")
files = [data[k * FILE : (k + 1) * FILE] for k in range(N_FILES)]
assert all(len(f) == FILE for f in files)
mb = N_FILES * FILE / 1e6


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


# warm-up: module loads, grow-only buffers, the decoder's graphs
w = codec.compress_many(model, [files[0][:700], files[1][:300]])
assert codec.decompress_many(model, w) == [files[0][:700], files[1][:300]] and codec.decompress(model, w[1]) == files[1][:300]
assert codec.compress(model, files[0][:700]) == w[0]

many, t_many = timed(lambda: codec.compress_many(model, files))
singles, t_singles = timed(lambda: [codec.compress(model, f) for f in files])
assert many == singles, "compress_many differs from compress"
res["compress"] = {
    "workload": f"{N_FILES} files x {FILE} B (enwik8 stand-in), SmolLM-135M random init seed 0, byte ids, 1 segment per file",
    "containers_identical": True,
    "container_bytes": sum(map(len, many)),
    "compress_many": {"s": t_many, "files_per_s": N_FILES / t_many, "MB_per_s": mb / t_many, "ms_per_file": 1e3 * t_many / N_FILES},
    "compress_loop": {"s": t_singles, "files_per_s": N_FILES / t_singles, "MB_per_s": mb / t_singles, "ms_per_file": 1e3 * t_singles / N_FILES},
    "speedup": t_singles / t_many,
}
print(json.dumps(res["compress"]), flush=True)

back, t_dmany = timed(lambda: codec.decompress_many(model, many))
assert back == files, "decompress_many did not return the inputs"
sub = list(range(n_single))
one, t_done = timed(lambda: [codec.decompress(model, many[i]) for i in sub])
assert one == [files[i] for i in sub]
per_single = t_done / len(sub)
res["decompress"] = {
    "decompress_many": {"files": N_FILES, "streams_per_wave": N_FILES, "s": t_dmany, "files_per_s": N_FILES / t_dmany, "MB_per_s": mb / t_dmany,
                        "ms_per_file": 1e3 * t_dmany / N_FILES},
    "decompress_loop": {"files": len(sub), "which": f"files {sub[0]}..{sub[-1]}", "s": t_done, "s_per_file": per_single,
                        "files_per_s": 1 / per_single, "MB_per_s": FILE / 1e6 / per_single,
                        "ms_per_token": 1e3 * per_single / FILE},
    "speedup_per_file": per_single / (t_dmany / N_FILES),
}
print(json.dumps(res["decompress"]), flush=True)
os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
with open(out_path, "w") as fh:
    json.dump(res, fh, indent=1)
print(f"wrote {out_path}")
