#!/bin/bash
# Round-2 GPU session driver: bash scripts/gpu_r2.sh <tag> <stage> [<stage> ...]
#   tests | bench | ref | tp (whole-step tensor-pipe ncu) | cfg (bench --config 1, 2 and SSD-1B b8) | launches | full
TAG=$1; shift
mkdir -p gpurun_out
for st in "$@"; do
case $st in
tests)
  timeout -k 10 1500 python -m pytest tests -m gpu -x -q -s > gpurun_out/tests_$TAG.log 2>&1; echo "tests rc=$?"; tail -5 gpurun_out/tests_$TAG.log;;
testsq)
  timeout -k 10 1500 python -m pytest tests -m gpu -x -q > gpurun_out/tests_$TAG.log 2>&1; echo "tests rc=$?"; tail -15 gpurun_out/tests_$TAG.log;;
smoke)
  timeout -k 10 600 python __graft_entry__.py smoke > gpurun_out/smoke_$TAG.log 2>&1; echo "smoke rc=$?"; tail -3 gpurun_out/smoke_$TAG.log;;
bench)
  timeout -k 10 1200 python bench.py > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err; echo "bench rc=$?"; tail -c 1500 gpurun_out/bench_$TAG.json; tail -3 gpurun_out/bench_$TAG.err;;
benchq)
  timeout -k 10 900 python bench.py --no-cpu-baseline > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err; echo "bench rc=$?"; tail -c 1500 gpurun_out/bench_$TAG.json; tail -3 gpurun_out/bench_$TAG.err;;
ref)
  timeout -k 10 900 python bench.py --impl reference --steps 2 > gpurun_out/ref_$TAG.json 2> gpurun_out/ref_$TAG.err; echo "ref rc=$?"; cat gpurun_out/ref_$TAG.json
  timeout -k 10 900 python bench.py --config 0 --steps 1 > gpurun_out/ref_cfg0_$TAG.json 2> gpurun_out/ref_cfg0_$TAG.err; echo "cfg0 rc=$?"; cat gpurun_out/ref_cfg0_$TAG.json;;
cfg)
  timeout -k 10 600 python bench.py --config 1 --steps 3 > gpurun_out/bench_cfg1_$TAG.json 2> gpurun_out/bench_cfg1_$TAG.err; echo "cfg1 rc=$?"; tail -c 800 gpurun_out/bench_cfg1_$TAG.json
  timeout -k 10 600 python bench.py --config 2 --steps 20 --no-cpu-baseline > gpurun_out/bench_cfg2_$TAG.json 2> gpurun_out/bench_cfg2_$TAG.err; echo "cfg2 rc=$?"; tail -c 800 gpurun_out/bench_cfg2_$TAG.json
  timeout -k 10 600 python bench.py --model ssd-1b --batch 8 --no-cpu-baseline > gpurun_out/bench_ssd1b_b8_$TAG.json 2> gpurun_out/bench_ssd1b_b8_$TAG.err; echo "ssd1b b8 rc=$?"; tail -c 800 gpurun_out/bench_ssd1b_b8_$TAG.json;;
tp)
  M=sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed,gpu__time_duration.sum
  timeout -k 10 900 python scripts/step_probe.py edit > gpurun_out/probe_$TAG.log 2>&1 &&
  timeout -k 10 1500 ncu --profile-from-start off --clock-control none --csv --log-file gpurun_out/tp_edit_$TAG.csv --metrics $M python scripts/step_probe.py edit > gpurun_out/tp_edit_$TAG.log 2>&1; echo "tp edit rc=$?"
  timeout -k 10 1500 ncu --profile-from-start off --clock-control none --csv --log-file gpurun_out/tp_unet_$TAG.csv --metrics $M python scripts/step_probe.py unet > gpurun_out/tp_unet_$TAG.log 2>&1; echo "tp unet rc=$?"
  python scripts/ncu_tensor_pipe.py gpurun_out/tp_edit_$TAG.csv gpurun_out/tp_unet_$TAG.csv > gpurun_out/${TAG}_tensor_pipe_step.json; head -c 900 gpurun_out/${TAG}_tensor_pipe_step.json;;
launches)
  CMD="python bench.py --steps 1 --warmup 3 --no-cpu-baseline"
  timeout -k 10 600 $CMD > gpurun_out/plain_$TAG.log 2>&1 &&
  timeout -k 10 1500 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_$TAG.csv --profile-from-start off python scripts/step_probe.py edit > gpurun_out/ncu_list_$TAG.log 2>&1; echo "launch list rc=$?";;
full)
  for K in gemm:k_gemm_conv:400:6 attn:'^k_attention_d64_p$':40:3 norm:'k_gn_apply|k_gn_stats':20:6 vaeattn:k_attn_vae:0:2; do
    IFS=: read name rx skip cnt <<< "$K"
    timeout -k 10 1500 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:"$rx" -s $skip -c $cnt -o gpurun_out/prof_${name}_$TAG -f python scripts/step_probe.py edit > gpurun_out/ncu_${name}_$TAG.log 2>&1; echo "ncu $name rc=$?"
  done;;
esac
done
ls gpurun_out | grep $TAG | head -40
