#!/usr/bin/env python3
"""bench.py -- the hot path's headline metric on B200: encode MB/s, SmolLM-135M, ctx 512 / reprime 512.

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU; N>1 under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port) on host cores
    python bench.py --sweep                                   # BASELINE config 5 table (chunk count 8..8192, low/high entropy)
    python bench.py --steps K --warmup W --dump-outputs DIR   # also writes the last timed step's payload / segment offsets as DIR/*.npy

Workload (BASELINE.json configs[1]): SmolLM-135M, 512 reprime-chunks batched on one B200, over enwik8.  Offline only the first
3 MiB of enwik8 exist (tests/golden/data/enwik8_3mib.xz = final_bench/enwik8_samples/enwik8_128kb_{0..23}); a "step" is one
pass of the hot path over ONE 262,144-byte slice of it per GPU (rank r takes slice r): 262,144 byte-level tokens -- no
tokenizer.json exists offline, so one token per byte, ids spread over the vocabulary like real SmolLM2 ids
(tests/golden/corpus.py::spread_map) -- coded as 32 independent segments = 512 reprime-chunks (511-token prefill + 512 coded
tokens each, except each segment's first), seeded random-init weights of the SmolLM2-135M architecture (no checkpoint offline).
  value    CUDA events on the library's stream around K steps of cz_encode_dev (token ids already in HBM), profiling OFF
  e2e      the public host-buffer call cz_encode (pinned host ids in, payload bytes out), wall clock
  roofline the tcgen05 GEMM family's algorithmic FLOPs / its CUDA-event time from a SEPARATE profiled pass
Chunks are independent, so N GPUs each take their own slice with no collective on the data path (weak scaling); the
`sharded` object is the strong-scaling companion: ONE fixed input (the whole 3 MiB) through candlezip_b200.sharding on all N
ranks, container assembled on rank 0, BLAKE3 of the container printed (identical for every N), decoded back and compared.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import corpus  # noqa: E402  (tests/golden/corpus.py: committed corpora, stdlib + numpy only)

METRIC = "encode_MB_per_s_smollm135m_ctx512"
V_SMOLLM = 49152
# dram__bytes_read + dram__bytes_write per launch under ncu --set full (profiles/ncu_summary_r02.md; 253k-row layer-wave launches):
# qkv+rope 763 MB, o-proj (+ fused norm operands) 1754 MB, gate/up 1063 MB, down (+ fused norm operands) 2267 MB; x60 launches each,
# plus the LM head: 51.5 GB of logits written and 0.31 bytes read per byte written (operand re-reads, 7.8 GB per 127k-column launch)
NCU_GEMM_TRAFFIC_BYTES_PER_STEP = int(60 * (763 + 1754 + 1063 + 2267) * 1e6 + 51.54e9 * (1 + 7.77 / 24.94))
MFLOP_PER_TOKEN = 551.0  # SURVEY 8d: trunk 423.84 + head 56.62 + attention 70.57 MFLOP per coded token at ctx 512 / reprime 512
TRUNK_PARAMS = 106_168_320  # matmul params per token position, SURVEY 8d
HEAD_PARAMS = 28_311_552
KV_BYTES_PER_DECODE_TOKEN = 17.67e6  # SURVEY 8d: 2 * 30 * 192 * 767 bf16 elements per stepwise token at the steady-state window
SLICE = 262144
WORKLOAD = ("enwik8 stand-in (first 3 MiB of enwik8 = final_bench/enwik8_samples/enwik8_128kb_0..23; enwik8.zst is not mounted offline), "
            "byte-level tokens (no tokenizer.json offline) with ids spread over the vocab (mean id/V 0.10, like the shipped SmolLM2 id traces), "
            "SmolLM-135M seeded random-init bf16 weights / fp32 accumulate, ctx 512 / reprime 512")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def enwik_slice_ids(k):
    """token ids of the k-th 262,144-byte slice of the enwik8 stand-in (12 slices)"""
    d = corpus.load("enwik8_3mib")
    k %= len(d) // SLICE
    return corpus.byte_ids(d[k * SLICE:(k + 1) * SLICE], V_SMOLLM, spread=True)


def dump_outputs(d, arrays, budget=64 << 20):
    """writes each array as d/<name>.npy: 64-bit integers as float64 (exact below 2^53), everything else as float32.  Each array gets
    an equal share of `budget` bytes; one larger than its share is replaced by a fixed sample of its elements (seed 0, ascending
    positions), so that two builds given the same arguments write files that compare element for element."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a).ravel()
        a = a.astype(np.float64 if a.dtype.itemsize == 8 else np.float32)
        keep = budget // len(arrays) // a.itemsize
        if a.size > keep:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(d, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1403.8), d.get("hbm_gbs", 6553.9), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples nvidia-smi clocks / throttle reasons DURING the timed region"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU reference (the oracle: C restatement of the reference's loop).  Nothing here imports candlezip_b200: the weights come from
# the numpy restatement of the product's seeded generator (tests/oracle_weights.py, asserted bit-equal in the CPU suite).
# ---------------------------------------------------------------------------------------------------------------------
class OracleSmolLM:
    def __init__(self):
        import oracle
        import oracle_weights as ow

        self.oracle = oracle
        self.cfg = dict(ow.SMOLLM_135M)
        self.sess = oracle.Session.llama(self.cfg, ow.smollm_random_init(self.cfg, 0, 0.02, 0.02), round_bf16=0, max_pos=1100)
        self.v = self.cfg["vocab"]
        self.cdf = np.empty(self.v + 1, np.uint32)

    def code_chunk(self, prime, targets, enc):
        """one steady-state reprime chunk (src/main.rs:2280-2350): fresh cache, prefill of `prime`, then per coded token
        to_vec1 + softmax_pdf + quantize_pdf_to_cdf + encode_counts + step"""
        o, lib = self.oracle, self.oracle.lib
        cdfp = self.cdf.ctypes.data_as(o.u32p)
        pa = np.ascontiguousarray(prime, np.uint32)
        logits = lib.czo_session_reprime(self.sess._h, pa.ctypes.data_as(o.u32p), len(pa))
        for s in targets:
            lib.czo_logits_to_cdf(logits, self.v, 0, cdfp)
            lib.czo_encoder_encode_counts(enc, int(self.cdf[s]), int(self.cdf[s + 1]), 1 << 30)
            logits = lib.czo_session_step_logits(self.sess._h, int(s))

    def time_chunk(self, seq, k):
        """times steady-state chunk k (>= 1) of the BOS-first sequence `seq`: returns (seconds, coded tokens)"""
        lib = self.oracle.lib
        i0 = 512 * k  # loop index of the chunk's first coded token (sym = seq[i0 + 1]); prime = seq[i0 + 1 - 511 .. i0 + 1)
        prime, targets = seq[i0 + 1 - 511:i0 + 1], seq[i0 + 1:i0 + 513]
        t0 = time.perf_counter()
        enc = lib.czo_encoder_new()
        self.code_chunk(prime, targets, enc)
        n = C.c_size_t()
        lib.czo_encoder_finish(enc, C.byref(n))
        lib.czo_encoder_free(enc)
        return time.perf_counter() - t0, len(targets)

    def encode_stream(self, ids):
        """the whole reference loop on one stream (BOS + ids): returns (seconds, payload bytes, n reprimes)"""
        t0 = time.perf_counter()
        payload, reprimes = self.sess.encode_tokens(np.concatenate([[0], ids]).astype(np.uint32))
        return time.perf_counter() - t0, payload, len(reprimes)


def run_reference(args):
    if env_int("RANK", 0) != 0:
        return
    orc = OracleSmolLM()
    seq = np.concatenate([[0], enwik_slice_ids(0)]).astype(np.uint32)  # rank 0's slice, as one BOS-first stream
    n_chunks = (len(seq) - 1) // 512
    for w in range(min(args.warmup, 1)):  # the CPU path has no warm-up effects worth minutes of wall clock
        orc.time_chunk(seq, 1)
    times, toks = [], 0
    for s in range(args.steps):
        dt, n = orc.time_chunk(seq, 1 + s % (n_chunks - 1))
        times.append(dt)
        toks += n
    t = sum(times)
    mbps = toks / t / 1e6
    sample = (f"{args.steps} steady-state reprime chunks of rank 0's enwik8 slice, one per step: 511-token prefill + 512 coded tokens each "
              f"(src/main.rs:2280-2350), oracle = C restatement of the reference loop, f32, OpenMP on {os.cpu_count()} cores")
    line = {
        "impl": "reference", "metric": METRIC, "value": mbps, "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "enwik8 stand-in (3 MiB), synthetic weights",
        "config": {"workload": WORKLOAD, "sample_tokens_per_step": 512, "prefill_tokens_per_step": 511, "bytes_per_token": 1,
                   "chunks_timed": args.steps},
        "cpu_baseline": {"value": mbps, "unit": "MB/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": mbps, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "tokens_per_s": toks / t,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
def schedule_work(model, _lib, seg_start):
    """teacher-forced rows and chunk count of a schedule (for FLOP accounting)"""
    first = np.zeros(4096, np.uint64); nc = np.zeros(4096, np.uint32); ps = np.zeros(4096, np.uint64); pl = np.zeros(4096, np.uint32)
    rows = n_chunks = 0
    for g in range(len(seg_start) - 1):
        k = _lib.lib.cz_schedule_chunks(int(seg_start[g + 1] - seg_start[g]), 512, 512, first.ctypes.data_as(_lib.u64p),
                                        nc.ctypes.data_as(_lib.u32p), ps.ctypes.data_as(_lib.u64p), pl.ctypes.data_as(_lib.u32p), 4096)
        rows += int((pl[:k].astype(np.int64) + nc[:k].astype(np.int64) - 1).sum())
        n_chunks += int(k)
    return rows, n_chunks


class Dist:
    """torch.distributed plumbing: NCCL for the barrier / max-over-ranks time, a gloo side group for python objects"""

    def __init__(self):
        import torch

        self.torch = torch
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        torch.cuda.set_device(self.local)
        self.dist = None
        self.gloo = None
        if self.world > 1:
            import torch.distributed as dist

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            # NCCL prints its version banner on STDOUT when the first communicator is created; stdout must carry exactly one JSON
            # line, so fd 1 points at stderr until the communicator exists
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
                dist.barrier()
                torch.cuda.synchronize()
                self.gloo = dist.new_group(backend="gloo")
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def bcast_obj(self, obj):
        if not self.dist:
            return obj
        lst = [obj]
        self.dist.broadcast_object_list(lst, src=0, group=self.gloo)
        return lst[0]

    class _ObjGroup:  # the `dist` argument of candlezip_b200.sharding: gather_object over the gloo side group
        def __init__(self, outer):
            self.o = outer

        def gather_object(self, obj, out, dst=0):
            self.o.dist.gather_object(obj, out, dst=dst, group=self.o.gloo)

    def obj_group(self):
        return self._ObjGroup(self) if self.dist else None

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def sharded_roundtrip(cz, model, D, data, ids, n_segments, vocab, spread):
    """ONE fixed input through candlezip_b200.sharding on all ranks (strong scaling): contiguous segment ranges per rank,
    Model.encode on each, payloads gathered to rank 0, container assembled there; then the container is broadcast, every
    rank decodes its range (Model.decode) and rank 0 compares the bytes.  Returns the result dict on rank 0 (None elsewhere)."""
    from candlezip_b200 import container, sharding

    enc = lambda part, seg: model.encode(part, seg_start=seg)[0]  # noqa: E731
    dec = lambda pays, seg: model.decode(pays, seg)  # noqa: E731
    grp = D.obj_group()
    sharding.encode_sharded(enc, ids, n_segments, D.rank, D.world, grp)  # warm-up at full size (grow-only buffers)
    D.barrier()
    t0 = time.perf_counter()
    pays, seg_start = sharding.encode_sharded(enc, ids, n_segments, D.rank, D.world, grp)
    blob = None
    if D.rank == 0:
        f = dict(token_count=len(ids), orig_len_bytes=len(data), vocab_size=vocab, orig_hash16=container.blake3_16(data))
        blob = container.write_container(f, b"random-init", pays, seg_tokens=np.diff(seg_start), engine=model.engine)
    D.barrier()
    enc_s = D.max(time.perf_counter() - t0)
    blob = D.bcast_obj(blob)
    _, _, _, _, st, payloads = container.read_container(blob)
    seg2 = np.concatenate([[0], np.cumsum(st)]).astype(np.uint64)
    D.barrier()
    t0 = time.perf_counter()
    out = sharding.decode_sharded(dec, payloads, seg2, D.rank, D.world, grp)
    D.barrier()
    dec_s = D.max(time.perf_counter() - t0)
    if D.rank != 0:
        return None
    ok = corpus.ids_to_bytes(out, vocab, spread) == data
    steps = int(max(np.diff(seg2)))
    return {"scaling": "strong", "input_bytes": len(data), "segments": int(len(seg2) - 1), "tokens_per_segment": steps,
            "encode_MB_per_s": len(data) / enc_s / 1e6, "decode_MB_per_s": len(data) / dec_s / 1e6, "encode_s": enc_s, "decode_s": dec_s,
            "decode_ms_per_step": 1e3 * dec_s / steps, "container_bytes": len(blob), "container_blake3_16": container.blake3_16(blob).hex(),
            "roundtrip_ok": bool(ok), "timing": "wall clock, barrier on both sides, max over ranks; includes gather + container assembly (encode)"}


def run_ours(args):
    import torch

    import candlezip_b200 as cz
    from candlezip_b200 import _lib, container

    D = Dist()
    rank, world, local = D.rank, D.world, D.local
    ctx = cz.Context(local)
    model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    n = args.tokens
    ids_host = torch.empty(n, dtype=torch.int32).pin_memory()
    ids_np = ids_host.numpy().view(np.uint32)
    ids_np[:] = np.resize(enwik_slice_ids(rank), n)
    seg_start = cz.split_segments(n, args.segments)
    sched, keep = model._schedule(n, seg_start, 0, 512, 512, None, 0)
    S = int(sched.n_segments)
    cap = 4 * n + 8 * S + 16
    rows, n_chunks = schedule_work(model, _lib, seg_start)
    gemm_flops = 2.0 * TRUNK_PARAMS * rows + 2.0 * HEAD_PARAMS * n

    # ---- device-resident arm (`value`): profiling OFF ----
    ids_dev = torch.empty(n, dtype=torch.int32, device="cuda")
    ids_dev.copy_(ids_host)
    out_dev = torch.empty(cap, dtype=torch.uint8, device="cuda")
    seg_off = np.zeros(S + 1, np.uint64)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr())

    def step_dev():
        _lib.check(_lib.lib.cz_encode_dev(model._h, C.c_void_p(ids_dev.data_ptr()), n, C.byref(sched), C.c_void_p(out_dev.data_ptr()), cap,
                                          seg_off.ctypes.data_as(_lib.u64p)))

    for _ in range(args.warmup):
        step_dev()
    D.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_dev()
    ev1.record(stream)
    D.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop()
    payload_bytes = int(seg_off[S])
    if args.dump_outputs:
        # what a caller of cz_encode_dev receives from the last timed step: the concatenated segment bitstreams and their offsets
        sfx = f"_rank{rank}" if world > 1 else ""
        dump_outputs(args.dump_outputs, {"payload" + sfx: out_dev[:payload_bytes].cpu().numpy(), "seg_off" + sfx: seg_off},
                     budget=(64 << 20) // world)
    ms_max = D.max(ms)
    value = world * n * args.steps / (ms_max / 1e3) / 1e6

    # ---- per-family device time: a SEPARATE pass with deferred CUDA-event pairs around every launch ----
    prof_steps = max(1, min(3, args.steps))
    ctx.profile(2)
    ctx.profile_read(reset=True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record(stream)
    for _ in range(prof_steps):
        step_dev()
    pe1.record(stream)
    D.barrier()
    prof_ms_per_step = pe0.elapsed_time(pe1) / prof_steps
    fam = ctx.profile_read(reset=True)
    ctx.profile(0)

    # ---- end-to-end arm through the public host-buffer API ----
    out_host = torch.empty(cap, dtype=torch.uint8).pin_memory()
    seg_off2 = np.zeros(S + 1, np.uint64)
    bs = _lib.Bitstreams(C.cast(out_host.data_ptr(), _lib.u8p), cap, seg_off2.ctypes.data_as(_lib.u64p))
    idp = C.cast(ids_host.data_ptr(), _lib.u32p)

    def step_e2e():
        _lib.check(_lib.lib.cz_encode(model._h, idp, n, C.byref(sched), C.byref(bs)))

    step_e2e()
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    D.barrier()
    e2e_value = world * n * args.steps / D.max(time.perf_counter() - t0) / 1e6
    same = bool(np.array_equal(seg_off, seg_off2)) and bool(torch.equal(out_dev[:payload_bytes].cpu(), out_host[:payload_bytes]))
    mean_sym_over_v = float(ids_np.astype(np.float64).mean() / V_SMOLLM)

    # ---- strong-scaling companion + decode at the headline config: the WHOLE 3 MiB through the sharded product path ----
    sharded = None
    if args.sharded_segments > 0:
        data = corpus.load("enwik8_3mib")[:args.sharded_bytes]
        sharded = sharded_roundtrip(cz, model, D, data, corpus.byte_ids(data, V_SMOLLM, True), args.sharded_segments, V_SMOLLM, True)
        if sharded:
            tok_s = sharded["decode_MB_per_s"] * 1e6
            _, hbm, _ = measured_peaks()
            sharded["decode_achieved_hbm"] = {"GB_per_s": tok_s / world * KV_BYTES_PER_DECODE_TOKEN / 1e9, "peak": hbm,
                                              "frac": tok_s / world * KV_BYTES_PER_DECODE_TOKEN / 1e9 / hbm,
                                              "bytes_per_token": KV_BYTES_PER_DECODE_TOKEN, "per_gpu": True}

    # ---- BASELINE config 1: alice29.txt self-test (single v2 stream encode; decode of a 64-segment container), rank 0 ----
    alice = None
    if args.alice and rank == 0:
        adata = corpus.load("alice29.txt")
        aids = corpus.byte_ids(adata, V_SMOLLM, True)
        model.encode(aids, n_segments=1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p1, s1 = model.encode(aids, n_segments=1)  # the reference's layout: one AC stream for the file
        t1 = time.perf_counter()
        f = dict(token_count=len(aids), orig_len_bytes=len(adata), vocab_size=V_SMOLLM, orig_hash16=container.blake3_16(adata))
        blob1 = container.write_container(f, b"random-init", p1)
        p64, s64 = model.encode(aids, n_segments=64)
        t2 = time.perf_counter()
        out = model.decode(p64, s64)
        t3 = time.perf_counter()
        alice = {"file": "alice29.txt (148,481 B LF copy, final_bench/cantrbry)", "tokens": len(aids), "encode_s_single_stream": t1 - t0,
                 "encode_MB_per_s_single_stream": len(adata) / (t1 - t0) / 1e6, "container_bytes_single_stream": len(blob1),
                 "bits_per_byte_random_init": 8.0 * len(blob1) / len(adata), "decode_segments": 64, "decode_s": t3 - t2,
                 "decode_MB_per_s": len(adata) / (t3 - t2) / 1e6, "roundtrip_ok": corpus.ids_to_bytes(out, V_SMOLLM, True) == adata,
                 "note": "random-init weights: bits/byte is not a compression figure; the size is compared with the CPU reference in cpu_baseline"}
    D.barrier()

    # ---- BASELINE config 4: the agentic gate scan replayed from the shipped asyoulik run (agent_cache.jsonl + proof.csv), rank 0 ----
    gate_scan = None
    if args.gate and rank == 0:
        from candlezip_b200 import gate

        gids = np.load(os.path.join(ROOT, "tests", "golden", "reference_fixtures.npz"))["run_asyoulik_syms"].astype(np.uint32)
        texts, calls, decisions, shipped = gate.load_replay(corpus.replay("asyoulik"))
        smap = corpus.spread_map(V_SMOLLM)
        tok = lambda text, mx: smap[np.frombuffer(text.encode("utf-8"), np.uint8)][:mx]  # noqa: E731
        jobs, plan = gate.plan_scan(gids, texts, tok, 512, 512)
        model.xe_bits(jobs[:64])  # warm-up (buffers)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bits = model.xe_bits(jobs)
        t1 = time.perf_counter()
        records, events, gate_rows = gate.decide(plan, bits, 512)
        gp, _ = model.encode(gids, n_segments=1, events=events or None)
        t2 = time.perf_counter()
        xe_rows = int(sum(len(p_) + len(t_) - 1 for p_, t_ in jobs))
        gate_scan = {"input": "asyoulik.txt as the shipped SmolLM2 token ids (39,915 ids, watchdog_decode_steps.jsonl) + the shipped agent_cache.jsonl "
                              "(30 agent texts, byte-level hint tokens: no tokenizer.json offline), --scan-lookahead 512, chunk 512",
                     "boundaries": len(plan), "xe_jobs": len(jobs), "xe_rows": xe_rows, "scan_s": t1 - t0, "xe_jobs_per_s": len(jobs) / (t1 - t0),
                     "xe_tokens_per_s": xe_rows / (t1 - t0), "gated": int(sum(r & 1 for r in records)), "gated_in_shipped_ledger": int(sum(g for g, _, _ in decisions.values())),
                     "encode_with_primes_s": t2 - t1, "payload_bytes": len(gp[0]),
                     "note": "all baseline / hint-conditioned passes of all 77 boundaries as ONE batch of paired streams (the reference runs them one after the "
                             "other on a second session, src/main.rs:2043-2054); random-init weights, so which hints gate is not comparable with the shipped ledger"}
    D.barrier()

    # ---- RWKV-7 0.1B (BASELINE config 3) on the enwik8 stand-in, sharded over the ranks; random-init weights ----
    rwkv = None
    if args.rwkv_bytes > 0:
        model.close()
        rmodel = cz.Model(ctx, cz.RWKV7_0P1B).random_init(0, 0.02, 0.02)
        rdata = corpus.load("enwik8_3mib")[:args.rwkv_bytes]
        ctx.profile(2)
        ctx.profile_read(reset=True)
        rwkv = sharded_roundtrip(cz, rmodel, D, rdata, corpus.byte_ids(rdata, 65536, True), args.rwkv_segments, 65536, True)
        rfam = ctx.profile_read(reset=True)
        ctx.profile(0)
        if rwkv:
            rwkv["model"] = "rwkv7-g1-0.1b shape (random-init), byte-level ids spread over V = 65536 (the trie tokenizer needs rwkv_vocab_v20230424.json, absent offline)"
        rmodel.close()

    if rank != 0:
        D.close()
        return
    peak_tf, peak_hbm, peak_src = measured_peaks()
    gemm_ms = fam["gemm"][0] / prof_steps
    achieved = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else None

    # per-kernel rooflines (DESIGN.md section 5): algorithmic flops or bytes of ONE step over the family's live device time
    cfgm = cz.SMOLLM_135M
    Dm, F, L, V = cfgm["d_model"], cfgm["d_ffn"], cfgm["n_layers"], cfgm["vocab"]
    qkv_n = Dm + 2 * cfgm["n_kv_heads"] * 64

    def kern(name, fam_key, bound, work):
        kms = fam[fam_key][0] / prof_steps
        if kms <= 0:
            return None
        if bound == "tensor":
            a, pk, unit = work / (kms / 1e3) / 1e12, peak_tf, "TFLOP/s"
        else:
            a, pk, unit = work / (kms / 1e3) / 1e9, peak_hbm, "GB/s"
        return {"kernel": name, "bound": bound, "achieved": a, "peak": pk, "unit": unit, "frac": a / pk, "ms_per_step": kms}

    kernels = [k for k in [
        kern("gemm_tc_kernel<256,SWIGLU,pair> gate/up", "gemm_gu", "tensor", 2.0 * rows * 2 * F * Dm * L),
        kern("gemm_tc_kernel<192,ADD_NORM_TMA,pair> down_proj (+ next norm's operands)", "gemm_down", "tensor", 2.0 * rows * Dm * F * L),
        # o_proj is bound by the fp32 residual: per row A 1152 B + residual read and written 4608 B + bf16 norm operand 1152 B
        kern("gemm_tc_kernel<192,ADD_NORM_TMA,pair> o_proj (+ next norm's operands)", "gemm_o", "hbm", float(rows) * (2 * Dm + 8 * Dm + 2 * Dm) * L),
        kern("gemm_tc_kernel<192,QKV_ROPE> qkv + RoPE", "gemm_qkv", "tensor", 2.0 * rows * qkv_n * Dm * L),
        kern("gemm_tc_kernel<256,COLMAX> LM head", "gemm_head", "tensor", 2.0 * HEAD_PARAMS * n),
        kern("attn_tc_kernel", "attn", "tensor", 70.57e6 * n),
        # CDF: one full read of the column for the sum (cdf_stats_tma_kernel, which also leaves e_v, v <= sym, in the e-cache) + the
        # prefix walk up to the coded symbol (cdf_bounds_warp_kernel): algorithmic 4V and 4V E[sym]/V bytes per token
        kern("cdf_stats_tma_kernel (max given by the LM head; sequential f64 sum; fills the e-cache)", "cdf", "hbm", 4.0 * V * n),
        kern("cdf_bounds_warp_kernel<cached> (prefix walk to the coded symbol)", "cdf_prefix", "hbm", 4.0 * V * n * mean_sym_over_v),
    ] if k]
    line = {
        "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "enwik8 stand-in (3 MiB), synthetic weights",
        "config": {"workload": WORKLOAD + f": {n} tokens per GPU per step (rank r codes 262,144-byte slice r) as {S} segments = {n_chunks} "
                               f"reprime-chunks ({rows} teacher-forced rows)",
                   "tokens_per_step_per_gpu": n, "segments": S, "chunks": n_chunks, "bytes_per_token": 1, "mean_symbol_id_over_vocab": mean_sym_over_v,
                   "l2": "per-step working set (about 3 GB of activations per wave + a 51.5 GB logits batch) exceeds the 126 MB L2 by orders of magnitude; no explicit flush",
                   "engine": "tcgen05", "value_timing": "CUDA events on the library's stream, profiling off"},
        "tokens_per_s": value * 1e6, "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "MB/s", "h2d_bytes_per_step": int(4 * n + 16 * rows + 4 * n),
                "d2h_bytes_per_step": int(payload_bytes + 8 * S + 16), "bitstream_equal_to_device_arm": same},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf if achieved else None,
                     # dram__bytes_read + dram__bytes_write per launch from the ncu --set full captures (profiles/), summed over one step
                     "traffic": NCU_GEMM_TRAFFIC_BYTES_PER_STEP, "traffic_source": "profiles/ncu_summary_r02.md (ncu --set full, per launch x launches per step)",
                     "kernel": "gemm_tc_kernel (tcgen05 GEMM family: qkv+rope/o/gate-up/down/lm_head; the RMSNorm passes live in the o/down epilogues)",
                     "flops_per_step": gemm_flops, "kernel_ms_per_step": gemm_ms, "peak_source": peak_src,
                     "timing": f"separate profiled pass ({prof_steps} steps, CUDA-event pairs around every launch, the CDF pass on the main stream instead of overlapped on the side stream; that pass ran at {prof_ms_per_step:.1f} ms/step)"},
        # whole-path tensor roofline exactly as SURVEY 8d defines it: tokens/s x 551.0 MFLOP / measured sustained bf16 peak
        "roofline_path": {"bound": "tensor", "achieved": value * 1e6 / max(1, world) * MFLOP_PER_TOKEN * 1e6 / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                          "frac": value * 1e6 / max(1, world) * MFLOP_PER_TOKEN * 1e6 / 1e12 / peak_tf, "per_gpu": True},
        "roofline_kernels": kernels,
        "kernel_ms_per_step": {k: v[0] / prof_steps for k, v in fam.items()},
        "kernel_launches_per_step": {k: v[1] // prof_steps for k, v in fam.items()},
        "compressed_bytes_per_step": payload_bytes, "sharded": sharded, "alice29": alice, "gate_scan": gate_scan, "rwkv7": rwkv,
    }
    if rwkv:
        rwkv["kernel_ms_total"] = {k: round(v[0], 2) for k, v in rfam.items()}
    if world == 1 and not args.no_cpu_baseline:
        # BASELINE.md section 3: the CPU reference on a >= 4,096-token prefix (>= 7 reprimes) of the config-1 file, the GPU path
        # on the same tokens beside it: encode MB/s and the compressed size (bits/byte parity, same weights, same input)
        model2 = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
        pre = corpus.byte_ids(corpus.load("alice29.txt")[:args.cpu_tokens], V_SMOLLM, True)
        gp, _ = model2.encode(pre, n_segments=1)
        model2.close()
        dt, payload, n_rep = OracleSmolLM().encode_stream(pre)
        line["cpu_baseline"] = {"value": len(pre) / dt / 1e6, "unit": "MB/s", "cores": os.cpu_count(), "kind": "port",
                                "sample": f"first {len(pre)} bytes of alice29.txt as one stream ({n_rep} reprimes, {dt:.1f} s): oracle = C restatement "
                                          "of the reference loop (src/main.rs:1979-2358), f32, OpenMP",
                                "compressed_bytes_cpu_ref": len(payload), "compressed_bytes_gpu": len(gp[0]),
                                "bits_per_byte_cpu_ref": 8.0 * len(payload) / len(pre), "bits_per_byte_gpu": 8.0 * len(gp[0]) / len(pre),
                                "size_rel_diff": (len(gp[0]) - len(payload)) / len(payload)}
    print(json.dumps(line), flush=True)
    D.close()


def run_sweep(args):
    """BASELINE config 5: synthetic byte streams (low entropy = the a-z cycle of final_bench/synthetic/alphabet.txt, high entropy =
    uniform bytes, PCG64 seed 0xC0FFEE), chunk count 8..8192 (one 512-token reprime chunk per segment-slot), encode MB/s per GPU."""
    import torch

    import candlezip_b200 as cz
    from candlezip_b200 import _lib

    D = Dist()
    ctx = cz.Context(D.local)
    model = cz.Model(ctx, cz.SMOLLM_135M).random_init(0, 0.02, 0.02)
    stream = torch.cuda.ExternalStream(ctx.stream_ptr())
    res = []
    for kind in ("low", "high"):
        for chunks in (8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192):
            n = chunks * 512
            data = corpus.low_entropy_stream(n) if kind == "low" else corpus.high_entropy_stream(n)
            ids = torch.from_numpy(corpus.byte_ids(data, V_SMOLLM, True).astype(np.int32)).cuda()
            segs = max(1, chunks // 16)  # 16 chunks per segment like the headline (8 -> one segment of 8 chunks)
            seg_start = cz.split_segments(n, segs)
            sched, keep = model._schedule(n, seg_start, 0, 512, 512, None, 0)
            cap = 4 * n + 8 * segs + 16
            out = torch.empty(cap, dtype=torch.uint8, device="cuda")
            off = np.zeros(segs + 1, np.uint64)
            step = lambda: _lib.check(_lib.lib.cz_encode_dev(model._h, C.c_void_p(ids.data_ptr()), n, C.byref(sched), C.c_void_p(out.data_ptr()),  # noqa: E731
                                                             cap, off.ctypes.data_as(_lib.u64p)))
            reps = 3 if chunks <= 1024 else 2
            step(); step()
            D.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                step()
            e1.record(stream)
            D.barrier()
            ms = D.max(e0.elapsed_time(e1)) / reps
            res.append({"entropy": kind, "chunks": chunks, "segments": segs, "tokens": n, "ms": ms, "MB_per_s_per_gpu": n / ms / 1e3,
                        "MB_per_s_total": D.world * n / ms / 1e3, "compressed_bytes": int(off[segs])})
    if D.rank == 0:
        print(json.dumps({"sweep": "BASELINE config 5 (synthetic streams, encode, SmolLM-135M random-init, ctx 512 / reprime 512)",
                          "n_gpus": D.world, "rows": res}), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--tokens", type=int, default=SLICE)
    ap.add_argument("--segments", type=int, default=32)
    ap.add_argument("--sharded-segments", type=int, default=1536,
                    help="segments of the whole-file strong-scaling / decode figure (1536 x 2048 tokens = 3 MiB: 3 reprimes per stream); 0 = skip")
    ap.add_argument("--sharded-bytes", type=int, default=3145728)
    ap.add_argument("--no-alice", dest="alice", action="store_false")
    ap.add_argument("--no-gate", dest="gate", action="store_false")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-tokens", type=int, default=4096, help="prefix of alice29.txt the CPU reference codes (>= 7 reprimes)")
    ap.add_argument("--rwkv-bytes", type=int, default=1048576, help="RWKV-7 figures on this prefix of the enwik8 stand-in (0 = skip)")
    ap.add_argument("--rwkv-segments", type=int, default=1024)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the payload bytes and segment offsets of the last timed step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.sweep or args.steps < 1):
        ap.error("--dump-outputs needs the default GPU arm and --steps >= 1")
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host core it can
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
        run_reference(args)
    elif args.sweep:
        run_sweep(args)
    else:
        os.environ.setdefault("OMP_NUM_THREADS", str(os.cpu_count() or 1)) if env_int("WORLD_SIZE", 1) == 1 else None
        run_ours(args)


if __name__ == "__main__":
    main()
