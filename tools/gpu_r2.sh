#!/bin/bash
# Round-2 development iteration on the GPU box: quick parity, per-workload timings.
cd "${GRAFT_REPO_ROOT:-/root/repo}"
mkdir -p gpurun_out
OUT=gpurun_out
PT="python -m pytest tests/test_gpu_parity.py -m gpu -q -x --timeout 300 -p no:cacheprovider"
timeout 600 $PT -k "${TESTK:-radix_sort or known_answers or small_random or edge}" > $OUT/pytest_quick.log 2>&1; echo "pytest quick rc=$?"; tail -n 3 $OUT/pytest_quick.log
for w in ${WL:-c2 c5 c3}; do timeout 300 python tools/profile_step.py $w 3 > $OUT/step_$w.log 2>&1; echo "$w rc=$?"; grep device_ms $OUT/step_$w.log | tail -n 1 | cut -c1-${CUT:-700}; grep -h parity $OUT/step_$w.log; done
if [ -n "$FULLTESTS" ]; then timeout 2400 $PT -k "${FULLK:-not 2147483648}" > $OUT/pytest_gpu.log 2>&1; echo "pytest full rc=$?"; tail -n 5 $OUT/pytest_gpu.log; fi
