#!/usr/bin/env python3
"""What the per-token code-length sinks (cz_model_set_code_length_out) cost on the encode path (GPU box only).
    python scripts/code_length_cost.py [out.json = profiles/code_length_r05.json] [steps = 6]
  encode   bench.py's headline step: SmolLM-135M seeded random init, the enwik8 stand-in's first 262,144 bytes as spread token ids
           (tests/golden/corpus.py::spread_map), 32 segments, cz_encode_dev; CUDA events around each step, profiling off.  Three settings
           alternated step by step after a warm-up of each: sinks off, intervals only (c_lo / c_hi), intervals plus entropy
  kernel   the entropy kernel alone: the `cdf` family's device time (deferred per-launch CUDA events, Context.profile(2)) with the entropy
           sink minus without it, per 131,072 columns; mode 0 and mode 2 (floored) on the headline step, mode 1 on the RWKV-7 step
  rwkv7    RWKV-7 0.1B shape, seeded random init, the stand-in's first 65,536 bytes spread over V = 65,536, 16 segments: encode step with
           and without the entropy sink, alternated
The GPU's name and power limit are read (query only) in the same run."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests", "golden")]
import candlezip_b200 as cz  # noqa: E402
import corpus  # noqa: E402
from candlezip_b200 import _lib  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "code_length_r05.json")
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 6
res = {"gpu": subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip(), "torch_device": torch.cuda.get_device_name(0)}
ctx = cz.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream_ptr())
data = corpus.load("enwik8_3mib")


def summary(x):
    x = np.asarray(x)
    return {"median": float(np.median(x)), "min": float(x.min()), "max": float(x.max()), "spread_pct": float(100 * (x.max() - x.min()) / np.median(x)),
            "all": [round(float(v), 3) for v in x]}


class Step:
    """one cz_encode_dev call of n tokens in S segments with the given sinks"""

    def __init__(self, model, ids, S):
        self.model, self.n, self.S = model, len(ids), S
        self.sched, self.keep = model._schedule(self.n, cz.split_segments(self.n, S), 0, 512, 512, None, 0)
        self.cap = 4 * self.n + 8 * S + 16
        self.ids_dev = torch.from_numpy(ids.astype(np.int64)).to(torch.int32).cuda()
        self.out_dev = torch.empty(self.cap, dtype=torch.uint8, device="cuda")
        self.seg_off = np.zeros(S + 1, np.uint64)
        self.lo, self.hi = np.zeros(self.n, np.uint32), np.zeros(self.n, np.uint32)
        self.ent = np.zeros(self.n, np.float64)

    def __call__(self, sinks, floor=0):
        m = self.model._h
        lo = self.lo.ctypes.data_as(_lib.u32p) if sinks else None
        hi = self.hi.ctypes.data_as(_lib.u32p) if sinks else None
        ent = self.ent.ctypes.data_as(_lib.f64p) if sinks == "entropy" else None
        _lib.check(_lib.lib.cz_model_set_code_length_out(m, lo, hi, ent, self.n if sinks else 0))
        _lib.check(_lib.lib.cz_model_set_pdf_floor(m, floor))
        try:
            _lib.check(_lib.lib.cz_encode_dev(m, C.c_void_p(self.ids_dev.data_ptr()), self.n, C.byref(self.sched), C.c_void_p(self.out_dev.data_ptr()),
                                              self.cap, self.seg_off.ctypes.data_as(_lib.u64p)))
        finally:
            _lib.check(_lib.lib.cz_model_set_code_length_out(m, None, None, None, 0))
        return int(self.seg_off[self.S])

    def timed(self, settings, n_steps):
        payload = {}
        for s in settings * 2:  # warm-up of every setting (grow-only buffers, module loads)
            payload[s] = self(*s)
        assert len(set(payload.values())) == len(set(s[1] for s in settings)), payload  # the sinks change no byte
        ms = {s: [] for s in settings}
        for _ in range(n_steps):
            for s in settings:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                assert self(*s) == payload[s]
                e1.record(stream)
                e1.synchronize()
                ms[s].append(e0.elapsed_time(e1))
        return ms, payload

    def cdf_family_ms(self, sinks, floor=0, reps=2):
        ctx.profile(2)
        ctx.profile_read(reset=True)
        for _ in range(reps):
            self(sinks, floor)
        torch.cuda.synchronize()
        fam = ctx.profile_read(reset=True)
        ctx.profile(0)
        return fam["cdf"][0] / reps, fam["cdf"][1] / reps


# ---- the headline step: off / intervals / intervals + entropy, alternated ----
model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
n, S = 262144, 32
step = Step(model, corpus.byte_ids(data[:n], 49152, True), S)
settings = [(None, 0), ("intervals", 0), ("entropy", 0)]
ms, payload = step.timed(settings, steps)
med_off = float(np.median(ms[settings[0]]))
res["encode"] = {"workload": f"{n} tokens (enwik8 stand-in, spread byte ids) as {S} segments per step, cz_encode_dev, SmolLM-135M random init",
                 "ms_per_step": {name: summary(ms[s]) for name, s in zip(("off", "intervals", "intervals_entropy"), settings)},
                 "over_off": {name: float(np.median(ms[s]) / med_off) for name, s in zip(("intervals", "intervals_entropy"), settings[1:])},
                 "payload_bytes": payload[settings[0]]}
# (mode 2, floored: off against intervals + entropy)
ms2, _ = step.timed([(None, 1), ("entropy", 1)], max(2, steps // 2))
res["encode_mode2"] = {"ms_per_step": {"off": summary(ms2[(None, 1)]), "intervals_entropy": summary(ms2[("entropy", 1)])}}

# ---- the entropy kernel alone, per 131,072 columns ----
kernel = {}
for floor, name in ((0, "mode0"), (1, "mode2")):
    base, nb = step.cdf_family_ms(None, floor)
    with_e, nw = step.cdf_family_ms("entropy", floor)
    kernel[name] = {"cdf_family_ms_off": round(base, 3), "cdf_family_ms_entropy": round(with_e, 3), "entropy_launches_per_step": int(nw - nb),
                    "ms_per_131072_columns": round((with_e - base) * 131072 / n, 3)}
model.close()

# ---- RWKV-7: encode step with and without the entropy sink ----
rmodel = cz.Model(ctx, cz.RWKV7_0P1B).random_init(0, 0.02, 0.02)
nr, Sr = 65536, 16
rstep = Step(rmodel, corpus.byte_ids(data[:nr], 65536, True), Sr)
rsettings = [(None, 0), ("entropy", 0)]
rms, rpay = rstep.timed(rsettings, max(2, steps // 2))
res["rwkv7_encode"] = {"workload": f"{nr} tokens (enwik8 stand-in, byte ids spread over V = 65,536) as {Sr} segments, cz_encode_dev, RWKV-7 0.1B random init",
                       "ms_per_step": {"off": summary(rms[rsettings[0]]), "intervals_entropy": summary(rms[rsettings[1]])},
                       "over_off": float(np.median(rms[rsettings[1]]) / np.median(rms[rsettings[0]]))}
base, nb = rstep.cdf_family_ms(None)
with_e, nw = rstep.cdf_family_ms("entropy")
kernel["mode1"] = {"cdf_family_ms_off": round(base, 3), "cdf_family_ms_entropy": round(with_e, 3), "entropy_launches_per_step": int(nw - nb),
                   "ms_per_131072_columns": round((with_e - base) * 131072 / nr, 3)}
res["entropy_kernel"] = {"method": "cdf family device time with the entropy sink minus without (deferred per-launch CUDA events), scaled to "
                                   "131,072 columns", **kernel}
rmodel.close()
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
json.dump(res, open(out_path, "w"), indent=1)
print(json.dumps(res, indent=1))
