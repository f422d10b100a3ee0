#!/bin/bash
mkdir -p gpurun_out
run() { local name=$1; shift; timeout 900 python -m pytest "$@" -x -q > gpurun_out/$name.log 2>&1; echo "$name exit=$? :: $(tail -n 1 gpurun_out/$name.log)"; }
run am tests/test_gpu_ops.py -k "argmax or ctc"
run fused tests/test_gpu_encoder.py tests/test_gpu_parity_full.py
grep -E "^(E |FAILED|ERROR)|assert|Error" gpurun_out/am.log gpurun_out/fused.log | head -n 20
timeout 300 python scripts/bench_ctc_fc.py 2>&1 | tee gpurun_out/bench_ctc_fc.txt
