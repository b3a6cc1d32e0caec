#!/bin/bash
# Outputs of the parent build (LIBBNR=variants/parent/libbnr.so) and of this tree, byte for byte, at configs 2-5; then
# the chain-group rule of the INT8 path re-measured at 8 and 12 chains with 1, 2 and 3 groups.
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r3}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r3_outputs_card.txt
Q="--steps 20 --warmup 2 --no-other-configs --no-strong --no-cpu-baseline --ess-burn 0 --ess-draws 0"
for cfg in c3 c5 c2 c4; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 200 python bench.py $Q --config $cfg --dump-outputs /tmp/dump_parent_$cfg > /dev/null 2>&1
  timeout 200 python bench.py $Q --config $cfg --dump-outputs /tmp/dump_new_$cfg > /dev/null 2>&1
  n=$(ls /tmp/dump_new_$cfg/*.npy | wc -l)
  if diff -r /tmp/dump_parent_$cfg /tmp/dump_new_$cfg > /dev/null && [ "$n" -gt 0 ]; then echo "$cfg: $n .npy files identical"
  else echo "$cfg: outputs DIFFER or missing ($n files)"; fi
done > $OUT/r3_outputs.txt
Q="--steps 100 --warmup 5 --no-other-configs --no-strong --no-cpu-baseline --ess-burn 0 --ess-draws 0"
for C in 8 12; do for g in 1 2 3; do
  echo -n "chains $C groups $g: "
  timeout 200 python bench.py $Q --chains $C --chain-groups $g 2>/dev/null | tail -1 | python -c "import json,sys; print(json.loads(sys.stdin.read())['ms_per_step'])"
done; done > $OUT/r3_groups.txt 2>&1
cat $OUT/r3_outputs_card.txt $OUT/r3_outputs.txt $OUT/r3_groups.txt
