#!/bin/bash
# Run each GPU test file in its own process (a trapped kernel poisons the CUDA context of its process
# only) and keep the logs under gpurun_out/.
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,driver_version,memory.total --format=csv | tee gpurun_out/gpu.txt
ls /root/reference 2>&1 | head -2
for f in ${@:-tests/test_gpu_sampler_step.py tests/test_gpu_groupnorm.py tests/test_gpu_simt.py tests/test_gpu_conv_tc.py tests/test_gpu_conv_halo.py tests/test_gpu_conv_halo_swap.py tests/test_gpu_attention_tc.py tests/test_gpu_model.py tests/test_gpu_parity_r2.py tests/test_gpu_dpm_solver.py tests/test_gpu_repaint.py tests/test_gpu_seeded_noise.py tests/test_gpu_continuous.py tests/test_gpu_continuous_dpm.py tests/test_gpu_continuous_repaint.py}; do
  n=$(basename $f .py)
  echo "=== $f"
  timeout 900 python -m pytest $f -q -m gpu --timeout 300 -x 2>&1 | tail -40 | tee gpurun_out/$n.log
done
