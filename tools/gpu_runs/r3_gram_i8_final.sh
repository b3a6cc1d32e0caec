#!/bin/bash
# bench.py with default arguments, parent build (LIBBNR=variants/parent/libbnr.so) and this tree alternated, three runs
# each; smoke(); the determinism check at every BASELINE shape.  The GPU test suite runs from r3_gram_i8_pytest.sh
# (python -m pytest tests -m gpu).
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r3}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r3_final_card.txt
for r in 1 2 3; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 200 python bench.py > $OUT/r3_bench_parent_$r.json 2> /dev/null
  timeout 200 python bench.py > $OUT/r3_bench_new_$r.json 2> /dev/null
done
for f in $OUT/r3_bench_{parent,new}_?.json; do
  python -c "import json; d = json.loads(open('$f').read().strip().splitlines()[-1]); o = d['other_configs']
print('$f', 'c3 %.3f ms/sweep, Gram %.3f ms' % (d['ms_per_step'], d['phases_ms']['syrk']),
      ' '.join('%s %.3f' % (k, o[k]['ms_per_sweep']) for k in sorted(o)))"
done > $OUT/r3_bench.txt
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r3_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/r3_smoke.log
timeout 250 bash tools/gpu_runs/r2_det.sh > $OUT/r3_det.log 2>&1
cat $OUT/r3_final_card.txt $OUT/r3_bench.txt; tail -2 $OUT/r3_smoke.log; cat $OUT/r3_det.log
