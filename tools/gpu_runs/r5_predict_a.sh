#!/bin/bash
# Predictions for new networks: the new GPU tests, the cost per sweep and of the pooled select (tools/predict_overhead.py,
# with tools/lab/pred_select_lab built as its header says) and smoke().
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r5}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r5_card.txt
timeout 600 python -m pytest tests/test_gpu_predict.py -m gpu -q -p no:cacheprovider -x > $OUT/r5_pytest_predict.log 2>&1; echo "pytest rc=$?" >> $OUT/r5_pytest_predict.log
timeout 400 python tools/predict_overhead.py --inline > $OUT/r5_overhead.txt 2>&1; echo "overhead rc=$?" >> $OUT/r5_overhead.txt
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r5_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/r5_smoke.log
cat $OUT/r5_card.txt; tail -25 $OUT/r5_pytest_predict.log; cat $OUT/r5_overhead.txt; tail -2 $OUT/r5_smoke.log
