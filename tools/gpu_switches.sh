#!/bin/bash
# The GPU parity, training-kernel edge, image / frame enlargement, host-pipeline and quality tests under
# every A/B switch of the library (the fallback kernels): each line must end in "passed" (tests
# that assert the default kernel selection skip themselves).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
T=${1:-switches}
: > gpurun_out/${T}_switches.txt
for e in "SRCNN_FUSED_IMPL=pl" "SRCNN_FUSED_IMPL=simt" "SRCNN_C5_IMPL=simt SRCNN_B3_IMPL=simt" \
         "SRCNN_GW_IMPL=simt SRCNN_D1_IMPL=simt" "SRCNN_D1_IMPL=separate SRCNN_E2E_GRAPH=0" \
         "SRCNN_TRAIN_HEAD=0 SRCNN_E2E_SUBBANDS=7 SRCNN_E2E_RAMPCAP=4"; do
  r=$(env $e timeout 600 python -m pytest tests/test_gpu_parity.py tests/test_train_tc_edges.py tests/test_upscale.py tests/test_upscale_frames.py tests/test_host_pipelines.py tests/test_quality.py tests/test_upscale_yuv420.py tests/test_upscale_yuv420_device.py tests/test_chroma_siting.py tests/test_upscale_yuv420p10.py -m gpu -q 2>&1 | tail -1)
  echo "$e: $r" | tee -a gpurun_out/${T}_switches.txt
done
