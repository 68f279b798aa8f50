#!/bin/bash
# Collects the round's measurement evidence on the GPU box: bench line, ncu launch list of the same command, and
# `ncu --set full` captures of the dominant kernels.  Usage: bash scripts/gpu_profile.sh <tag>   (outputs -> gpurun_out/)
TAG=${1:-r1}
mkdir -p gpurun_out
CMD="python bench.py --steps 1 --warmup 3 --no-cpu-baseline"
# full default bench (with cpu_baseline) — the number that is reported
timeout -k 10 900 python bench.py > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err
echo "bench rc=$?"; tail -c 600 gpurun_out/bench_$TAG.json
# launch list: skip the 3 warm-up steps, capture one timed step's launches
timeout -k 10 600 $CMD > gpurun_out/plain_$TAG.log 2>&1 &&
NL=$(python -c "import json,sys; print(json.loads(open('gpurun_out/plain_$TAG.log').read().strip().splitlines()[-1])['gpu_launches'])") &&
echo "launches per step: $NL" &&
timeout -k 10 1200 ncu --metrics gpu__time_duration.sum --clock-control none -s $((3 * NL)) -c $NL --csv \
    --log-file gpurun_out/launches_$TAG.csv $CMD > gpurun_out/ncu_list_$TAG.log 2>&1
echo "ncu list rc=$?"
# full captures of the dominant kernels (inside the 4th step = the timed one); -s counts launches that match -k
NG=$(python -c "import json,sys; print(json.loads(open('gpurun_out/plain_$TAG.log').read().strip().splitlines()[-1])['roofline']['launches_per_step'])")
timeout -k 10 600 $CMD > gpurun_out/plain2_$TAG.log 2>&1 &&
timeout -k 10 1200 ncu --set full --clock-control none --import-source on -k regex:k_gemm_conv -s $((NG * 3 + 300)) -c 6 \
    -o gpurun_out/prof_gemm_$TAG -f $CMD > gpurun_out/ncu_gemm_$TAG.log 2>&1
echo "ncu gemm rc=$?"
timeout -k 10 600 $CMD > gpurun_out/plain3_$TAG.log 2>&1 &&
timeout -k 10 1200 ncu --set full --clock-control none --import-source on -k regex:'^k_attention_d64_p$' -s $((3 * 160 + 40)) -c 3 \
    -o gpurun_out/prof_attn_$TAG -f $CMD > gpurun_out/ncu_attn_$TAG.log 2>&1
echo "ncu attention rc=$?"
timeout -k 10 1200 ncu --set full --clock-control none --import-source on -k regex:'k_gn_apply|k_gn_stats' -s $((3 * 300 + 20)) -c 6 \
    -o gpurun_out/prof_norm_$TAG -f $CMD > gpurun_out/ncu_norm_$TAG.log 2>&1
echo "ncu norm rc=$?"
ls -la gpurun_out | tail -20
