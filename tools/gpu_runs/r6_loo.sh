#!/bin/bash
# Build, the PSIS-LOO tests, tools/loo_overhead.py, smoke, bench.py, then the whole suite.  Logs in $OUT.
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r6}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1 || { tail -20 $OUT/build.txt; exit 1; }
timeout 900 python -m pytest -q -x tests/test_gpu_loo.py > $OUT/pytest_loo.txt 2>&1; echo "loo tests rc=$?"
tail -15 $OUT/pytest_loo.txt
timeout 600 python tools/loo_overhead.py > $OUT/loo_overhead.txt 2>&1; echo "overhead rc=$?"
cat $OUT/loo_overhead.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; echo "smoke rc=$?"
tail -2 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 3 > $OUT/bench.txt 2>&1; echo "bench rc=$?"
tail -1 $OUT/bench.txt | cut -c1-400
timeout 1500 python -m pytest -q tests > $OUT/pytest_all.txt 2>&1; echo "suite rc=$?"
tail -15 $OUT/pytest_all.txt
