#!/bin/bash
# Run the GPU parity tests function by function in separate processes (a device-side trap poisons the CUDA
# context of its process), keeping the log under gpurun_out/.  Optional argument: an egrep filter on test names.
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
filter="${1:-.}"
mapfile -t groups < <(python -m pytest tests/test_engine_gpu.py tests/test_kernel_edges_gpu.py --collect-only -q -m gpu \
  -p no:cacheprovider 2>/dev/null \
  | grep "::" | sed 's/\[.*//' | sort -u | grep -E "$filter")
rc=0
: > gpurun_out/gpu_tests.log
rm -f gpurun_out/parity_stats.jsonl
for g in "${groups[@]}"; do
  echo "=== $g" >> gpurun_out/gpu_tests.log
  t0=$(date +%s)
  timeout 900 python -m pytest "$g" -q -m gpu --no-header -p no:cacheprovider >> gpurun_out/gpu_tests.log 2>&1 || rc=1
  echo "--- $(( $(date +%s) - t0 )) s" >> gpurun_out/gpu_tests.log
done
grep -E "^(===|---|[0-9]+ (passed|failed)|FAILED|ERROR|E  )" gpurun_out/gpu_tests.log | head -120
exit $rc
