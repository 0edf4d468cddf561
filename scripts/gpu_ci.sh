#!/bin/bash
# Runs the GPU suite in groups, each under its own timeout, logs into gpurun_out/ (used via gpurun).
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/gpu.txt 2>&1
run() { # name timeout pytest-args...
  local name=$1 t=$2; shift 2
  echo "=== $name" | tee -a gpurun_out/summary.txt
  timeout "$t" python -m pytest tests -m gpu -q -x "$@" > "gpurun_out/$name.log" 2>&1
  echo "exit=$? $(tail -n 1 gpurun_out/$name.log)" | tee -a gpurun_out/summary.txt
}
rm -f gpurun_out/summary.txt
run coder_cdf 600 -k "k1 or k2 or k3 or k9"
run gemm_simt 300 -k "gemm and simt"
run gemm_tc 300 -k "gemm and not simt"
run tiny_simt 900 -k "tiny and simt and not rwkv7_deep"
run tiny_tc 900 -k "tiny and not simt and not rwkv7_deep"
run full 900 -k "full_size and not rwkv7_deep"
run dictionary 900 -k "dictionary"
run match 1200 -k "match"
run rwkv 900 -k "((rwkv7 and not full_size) or hint_prime or gate_scan or file_level or cli_twin) and not rwkv7_deep"
run rwkv_deep 1200 -k "rwkv7_deep"
for f in gpurun_out/*.log; do echo "---- $f"; tail -n 25 "$f"; done
