#!/bin/bash
# Runs the GPU parity suite in separate processes (a trapped kernel poisons only its own process).
mkdir -p gpurun_out
export PYTHONUNBUFFERED=1
run() { name=$1; shift; echo "=== $name"; timeout 600 python -m pytest "$@" -q -m gpu -p no:cacheprovider > gpurun_out/$name.log 2>&1; echo "exit $?"; tail -n 3 gpurun_out/$name.log; }
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/smi.txt 2>&1
run rowops tests/test_kernels_gpu.py -k "not gemm"
run gemm_simt tests/test_kernels_gpu.py -k "(gemm_layouts and (True-1 or False-1)) or fp32_simt or (gemm_epilogues and (cdtype0-1 or cdtype1-1))"
for lay in "False-True" "False-False" "True-False" "True-True"; do
  run gemm_tc_$lay tests/test_kernels_gpu.py -k "gemm_layouts and $lay-2"
done
run gemm_tc_epi tests/test_kernels_gpu.py -k "gemm_epilogues and (cdtype0-2 or cdtype1-2)"
run gemm_tc_big tests/test_kernels_gpu.py -k "large_k or cta_pair"
run relattn tests/test_relattn_gpu.py
run bert_attn tests/test_bert_attn_gpu.py
run model tests/test_model_gpu.py
run requests tests/test_generate_requests_gpu.py
run requests_prefill tests/test_generate_requests_prefill_gpu.py
