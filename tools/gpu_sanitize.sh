#!/bin/bash
# compute-sanitizer memcheck over smoke() (every kernel family, small shapes); "full" adds the GPU test suite
set +e
mkdir -p gpurun_out
timeout 1200 compute-sanitizer --tool memcheck --print-limit 20 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/sanitize_smoke.log 2>&1; echo "memcheck smoke rc=$?"; grep -E "ERROR SUMMARY|smoke ok|Invalid|error" gpurun_out/sanitize_smoke.log | head -10
if [ "$1" = full ]; then
  timeout 900 compute-sanitizer --tool memcheck --print-limit 20 python -m pytest tests -m gpu -q -k "not c3_shape and not c5_shape and not full_size and not no_host_round_trip and not no_host_staging" > gpurun_out/sanitize_pytest.log 2>&1; echo "memcheck pytest rc=$?"; grep -E "ERROR SUMMARY|passed|failed|Invalid" gpurun_out/sanitize_pytest.log | head -8
fi
