#!/bin/bash
# Run the GPU parity suite file by file, each under its own timeout and process (a kernel trap
# poisons only that process).  Logs land in gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/smi.txt 2>&1
run() { # name, args...
  local name=$1; shift
  timeout 600 python -m pytest "$@" -x -q > gpurun_out/$name.log 2>&1
  echo "$name exit=$? :: $(tail -n 1 gpurun_out/$name.log)"
}
run gemm tests/test_gpu_ops.py -k "linear"
if ! grep -q passed gpurun_out/gemm.log || grep -q failed gpurun_out/gemm.log; then
  timeout 300 python scripts/debug_gemm.py > gpurun_out/debug_gemm.log 2>&1
  tail -n 40 gpurun_out/debug_gemm.log
fi
run small tests/test_gpu_ops.py -k "layernorm or cmvn or fc3_weight or row_stats"
run ctc tests/test_gpu_ops.py -k "ctc"
run conv tests/test_gpu_ops.py -k "conv_stack"
run attn tests/test_gpu_ops.py -k "attention"
run attn_edges tests/test_attention_edges.py
run attn_train_edges tests/test_attention_train_edges.py
run encoder tests/test_gpu_encoder.py
run misc tests/test_gpu_ops.py -k "custom_ops or collater"
run criterion tests/test_gpu_criterion.py
for f in gemm small ctc conv attn encoder misc criterion; do echo "=== $f"; grep -E "^(E |FAILED|ERROR)|assert|Error" gpurun_out/$f.log | head -n 12; done
