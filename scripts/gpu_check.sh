#!/bin/bash
# Runs the GPU test-suite in isolated processes (a trapped kernel poisons its CUDA context) with hard timeouts.
# Usage (on the GPU box): bash scripts/gpu_check.sh [pytest -k expressions...]
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu_info.txt 2>&1
run() { # name, pytest args...
  local name=$1; shift
  echo "=== $name" | tee -a gpurun_out/gpu_check.log
  timeout -k 10 600 python -m pytest -x -q -m gpu -p no:cacheprovider "$@" > gpurun_out/test_$name.log 2>&1
  local rc=$?
  tail -n 25 gpurun_out/test_$name.log | tee -a gpurun_out/gpu_check.log
  echo "=== $name rc=$rc" | tee -a gpurun_out/gpu_check.log
}
: > gpurun_out/gpu_check.log
run canny tests/test_gpu_canny.py
run elementwise tests/test_gpu_kernels.py -k "pre_post or test_silu or sincos or groupnorm or layernorm or softmax or scheduler or cin4"
run gemm_plain tests/test_gpu_kernels.py -k "gemm_plain"
run gemm_epi tests/test_gpu_kernels.py -k "gemm_epilogue or folded_layernorm"
run gemm_geglu tests/test_gpu_kernels.py -k "gemm_geglu"
run conv tests/test_gpu_kernels.py -k "test_conv3x3 and not cin4"
run attention tests/test_gpu_kernels.py -k "attention"
run guards tests/test_gpu_kernels.py -k "writes_only or write_only"
run engine tests/test_gpu_engine.py -s
run fullsize tests/test_gpu_fullsize.py -s
run dropin tests/test_gpu_dropin.py
run text_encoder tests/test_gpu_text_encoder.py -s
for extra in "$@"; do run extra tests -k "$extra"; done
grep -E "^=== .* rc=" gpurun_out/gpu_check.log
