#!/bin/bash
cd "$(dirname "$0")/.." || exit 1
mkdir -p gpurun_out; O=gpurun_out
timeout 900 python -m pytest tests/test_join_gpu.py tests/test_topk_gpu.py tests/test_forward_gpu.py -m gpu -x -q > $O/r02b_tests.log 2>&1; echo "pytest exit $?" >> $O/r02b_tests.log; tail -4 $O/r02b_tests.log
