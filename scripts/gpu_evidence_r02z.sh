#!/bin/bash
# Evidence visit for the wide attention kernel: bench line + launch list, ncu --set full of the attention kernel
# inside a step, timeline of CTA 0
TAG=${1:-r02z}
mkdir -p gpurun_out
bash scripts/gpu_bench_launches.sh $TAG
timeout 600 ncu --set full --clock-control none --import-source on --profile-from-start off \
  -k "regex:attention_fwd" -s 0 -c 1 -f -o gpurun_out/${TAG}_attention python scripts/profile_step.py > gpurun_out/${TAG}_attention.log 2>&1
echo "ncu attention exit=$?"
bash scripts/gpu_ab_variants.sh "timeout 200 python scripts/trace_attn.py" awtrace > gpurun_out/${TAG}_attention_timeline.txt 2>&1
