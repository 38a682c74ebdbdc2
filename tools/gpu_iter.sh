#!/bin/bash
# One development iteration on the GPU box: full GPU tests, per-workload timings.
cd "${GRAFT_REPO_ROOT:-/root/repo}"
mkdir -p gpurun_out
OUT=gpurun_out
timeout 1200 python -m pytest tests/test_gpu_parity.py -m gpu -q -x --timeout 600 -p no:cacheprovider -k "${TESTK:-not 2147483648}" > $OUT/pytest_gpu.log 2>&1; echo "pytest rc=$?"; tail -n 5 $OUT/pytest_gpu.log
for w in ${WL:-c2 c3 c5 c1}; do timeout 300 python tools/profile_step.py $w 3 > $OUT/step_$w.log 2>&1; echo "$w rc=$?"; grep device_ms $OUT/step_$w.log | tail -n 1 | cut -c1-${CUT:-900}; grep -h parity $OUT/step_$w.log; done
