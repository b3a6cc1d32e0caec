#!/bin/bash
# bench.py with default arguments, parent build (LIBBNR=variants/parent/libbnr.so) and this tree alternated, three runs
# each.  The GPU test suite runs from r4_gram_slice_pytest.sh; outputs, smoke(), the determinism check and the timeline
# from r4_gram_slice_outputs.sh.
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r4}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r4_final_card.txt
for r in 1 2 3; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 200 python bench.py > $OUT/r4_bench_parent_$r.json 2> /dev/null
  timeout 200 python bench.py > $OUT/r4_bench_new_$r.json 2> /dev/null
done
for f in $OUT/r4_bench_{parent,new}_?.json; do
  python -c "import json; d = json.loads(open('$f').read().strip().splitlines()[-1]); o = d['other_configs']
print('$f', 'c3 %.3f ms/sweep, Gram %.3f ms' % (d['ms_per_step'], d['phases_ms']['syrk']),
      ' '.join('%s %.3f' % (k, o[k]['ms_per_sweep']) for k in sorted(o)))"
done > $OUT/r4_bench.txt
cat $OUT/r4_final_card.txt $OUT/r4_bench.txt
