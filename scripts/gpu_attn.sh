#!/bin/bash
# one-pass attention visit: parity (attention ops, encoder, full-depth parity), NT wgrad, micro-benchmark
mkdir -p gpurun_out
run() { local name=$1; shift; timeout 900 python -m pytest "$@" -x -q > gpurun_out/$name.log 2>&1; echo "$name exit=$? :: $(tail -n 1 gpurun_out/$name.log)"; }
run attn tests/test_gpu_ops.py -k "attention"
run wgrad_nt tests/test_gpu_train_ops.py -k "wgrad"
run encoder tests/test_gpu_encoder.py
grep -E "^(E |FAILED|ERROR)|assert|Error" gpurun_out/attn.log gpurun_out/encoder.log gpurun_out/wgrad_nt.log | head -n 20
echo "=== one-pass"; timeout 300 python scripts/bench_attn.py 10 2>&1 | tee gpurun_out/bench_attn_onepass.txt
