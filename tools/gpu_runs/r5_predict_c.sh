#!/bin/bash
# Outputs of the parent build (LIBBNR=variants/parent/libbnr.so) and of this tree byte for byte at configs 2-5, then
# bench.py with default arguments, parent and this tree alternated, two runs each.
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r5}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r5_c_card.txt
Q="--steps 20 --warmup 2 --no-other-configs --no-strong --no-cpu-baseline --ess-burn 0 --ess-draws 0"
D=$(mktemp -d)
for cfg in c3 c5 c2 c4; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 200 python bench.py $Q --config $cfg --dump-outputs $D/parent_$cfg > /dev/null 2>&1
  timeout 200 python bench.py $Q --config $cfg --dump-outputs $D/new_$cfg > /dev/null 2>&1
  n=$(ls $D/new_$cfg/*.npy | wc -l)
  if diff -r $D/parent_$cfg $D/new_$cfg > /dev/null && [ "$n" -gt 0 ]; then echo "$cfg: $n .npy files identical"
  else echo "$cfg: outputs DIFFER or missing ($n files)"; fi
done > $OUT/r5_outputs.txt
rm -rf "$D"
for r in 1 2; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 150 python bench.py > $OUT/r5_bench_parent_$r.json 2> /dev/null
  timeout 150 python bench.py > $OUT/r5_bench_new_$r.json 2> /dev/null
done
for f in $OUT/r5_bench_{parent,new}_?.json; do
  python -c "import json; d = json.loads(open('$f').read().strip().splitlines()[-1]); o = d['other_configs']
print('$f', 'c3 %.3f ms/sweep' % d['ms_per_step'], ' '.join('%s %.3f' % (k, o[k]['ms_per_sweep']) for k in sorted(o)))"
done > $OUT/r5_bench.txt 2>&1
cat $OUT/r5_c_card.txt $OUT/r5_outputs.txt $OUT/r5_bench.txt
