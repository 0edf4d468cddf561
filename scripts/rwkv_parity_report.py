#!/usr/bin/env python3
"""Measures the RWKV-7 tolerances on the GPU box and writes the tables kept in profiles/rwkv_parity_rNN.md.

    python scripts/rwkv_parity_report.py > profiles/rwkv_parity_rNN.md

Kernel level: the WKV-7 scan and the LayerNorm-mix hooks against the f64 restatement (tests/rwkv7_ref.py), on the cases of
tests/test_gpu_rwkv7_deep.py.  Model level: every position of BOS-started runs, max|logit_gpu - logit_oracle| / std(oracle logits
of that position), against the oracle with the same bf16 rounding points and against the pure-f32 oracle, with the oracle against
itself (the rounding points alone) beside them.  TEST INFRASTRUCTURE: uses the oracle as the checker."""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import candlezip_b200 as cz  # noqa: E402
import test_gpu_rwkv7_deep as deep  # noqa: E402
from candlezip_b200 import _lib  # noqa: E402

ENGINE = {_lib.CZ_ENGINE_TCGEN05: "tcgen05", _lib.CZ_ENGINE_SIMT: "simt"}


def blocks(r, n=512):
    return " ".join(f"{r[i:i + n].max():.3g}" for i in range(0, len(r), n))


def scan_section(ctx):
    print("## WKV-7 scan against f64 (4,096 rows of one stream, every row class of scan_case)\n")
    print("per row: max over the row of (|out - ref| - ulp_bf16(ref) / 2)+ / std(ref row), the error beyond the bf16 rounding of the output\n")
    print("| H | layer0 | initial state | max over rows | mean | max per 512-row block | final state max|dS|/max|S| |")
    print("|---|---|---|---|---|---|---|")
    worst_row, worst_state = 0.0, 0.0
    for H, layer0, init in deep.SCAN_SHAPES:
        r = deep.scan_vs_f64(ctx, H, layer0, init)
        worst_row, worst_state = max(worst_row, r["row"].max()), max(worst_state, r["state"])
        print(f"| {H} | {layer0} | {'non-zero' if init else 'zero'} | {r['row'].max():.2e} | {r['row'].mean():.2e} | {blocks(r['row'])} | {r['state']:.3e} |")
    print(f"\n**scan vs f64, max over rows: {worst_row:.2e}; final state: {worst_state:.3e}**\n")


def ln_mix_section(ctx):
    print("## LayerNorm-mix against f64 (form 0: what the model runs; 1: the element-per-lane kernel forced)\n")
    print("bound: max |out - bf16(ref)| / (1 bf16 ulp + 2^-20 cond (|xn| + |prev|)), must be <= 1 (see ln_mix_metrics)\n")
    print("| C | nmix | state buffers | form | kernel (elements per lane) | bound, plain rows | share equal | bound, edge rows | "
          "state_out rel. err, plain rows | edge rows / cond |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    worst = {}
    for Cw in deep.LN_MIX_WIDTHS:
        for nmix in (1, 6):
            for in_place in (False, True):
                for form, used, m, kept in deep.ln_mix_run_case(ctx, Cw, nmix, in_place):
                    for k, v in m.items():
                        worst[k] = min(worst.get(k, 1.0), v) if k == "equal" else max(worst.get(k, 0.0), v)
                    print(f"| {Cw} | {nmix} | {'in place' if in_place else 'ping-pong'} | {form} | {used} | {m['bound']:.3f} | {m['equal']:.5f} | "
                          f"{m['edge_bound']:.3f} | {m['state']:.2e} | {m['state_edge']:.2e} |" + ("" if kept else " **unwritten slot changed**"))
    print(f"\n**LN-mix extremes: {worst}**\n")


def model_section(ctx):
    print("## Every position of a BOS-started run against the oracle\n")
    print("| configuration | engine | positions | reference | max over positions >= 1 | position 0 | mean | max per 512-position block |")
    print("|---|---|---|---|---|---|---|---|")
    cases = [(name, cfg, mk, engines, n, lit, 40 + i) for i, (name, cfg, mk, engines, n, lit) in enumerate(deep.deep_configs())]
    cases.append(deep.FULL_CONFIG + (50,))
    for name, cfg, mk, engines, n, lit, seed in cases:
        t0 = time.time()
        W = mk()
        targets = deep.deep_targets(cfg["vocab"], n, seed, lit)
        w16, w32 = deep.oracle_logits(cfg, W, targets)
        for eng in engines:
            model = deep.load(ctx, cfg, W, eng)
            r16, r32, rr = deep.parity(model.chunk_logits([0], targets), w16, w32)
            model.close()
            label = f"{name}" + (f", {lit:.0%} literal escapes" if lit else "")
            for ref, r in (("oracle, bf16 rounding points", r16), ("oracle, pure f32", r32), ("(oracle bf16 vs oracle f32)", rr)):
                print(f"| {label} | {ENGINE[eng]} | {n} | {ref} | **{r[1:].max():.5f}** (pos {1 + int(r[1:].argmax())}) | {r[0]:.5f} | "
                      f"{r.mean():.5f} | {blocks(r)} |")
                label = ""
        print(f"| | | | ({time.time() - t0:.0f} s with the CPU oracle; std(logits) at position 0 {w32[0].std():.4f}, "
              f"mean over positions {w32.std(axis=1).mean():.4f}) | | | | |")
    print()


def bits_section(ctx):
    print("## Bits per token on text sampled from the model (no reprime)\n")
    print("| configuration | lm_head scale | tokens | GPU payload bytes | oracle payload bytes | difference | oracle bits/token | log2 V |")
    print("|---|---|---|---|---|---|---|---|")
    for name, cfg, mk, scale, n, seed in (("RWKV7_TINY seed 7", deep.RWKV7_TINY, lambda: deep.make_weights(deep.RWKV7_TINY, 7), 2.0, 2000, 61),
                                           ("0.1B shape", cz.RWKV7_0P1B, lambda: deep.make_weights(cz.RWKV7_0P1B, 3), 2.0, 1024, 62)):
        got, ref, bpt, log2v = deep.bits_per_token_case(ctx, cfg, mk(), scale, n, seed)
        print(f"| {name} | {scale} | {n} | {got} | {ref} | {100.0 * (got - ref) / ref:+.2f} % | {bpt:.3f} | {log2v:.2f} |")
    print()


def main():
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    ctx = cz.Context(0)
    print("# RWKV-7 parity, measured on the GPU (scripts/rwkv_parity_report.py)\n")
    print(f"GPU: {gpu} (name, power limit, max SM clock)\n")
    for section in (scan_section, ln_mix_section, model_section, bits_section):
        t0 = time.time()
        try:
            section(ctx)
        except Exception as e:  # one failing section must not hide the others' numbers
            print(f"\n**{section.__name__} failed: {type(e).__name__}: {e}**\n")
        print(f"_{section.__name__}: {time.time() - t0:.0f} s_\n")
        sys.stdout.flush()


if __name__ == "__main__":
    main()
