#!/bin/bash
# The whole GPU test suite in two halves (each under ten minutes): bash r5_predict_b.sh a|b
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r5}"   # where the logs go
mkdir -p "$OUT"
A="tests/test_gpu_large_dims.py tests/test_gpu_engine.py tests/test_gpu_fit.py tests/test_gpu_multirank.py"
B=$(ls tests/test_gpu_*.py tests/test_multirank_gloo.py | grep -v -F -e large_dims -e gpu_engine -e gpu_fit -e gpu_multirank)
if [ "$1" = a ]; then F="$A"; else F="$B"; fi
timeout 570 python -m pytest $F -m gpu -q -p no:cacheprovider > $OUT/r5_pytest_$1.log 2>&1; echo "pytest rc=$?" >> $OUT/r5_pytest_$1.log
tail -15 $OUT/r5_pytest_$1.log
