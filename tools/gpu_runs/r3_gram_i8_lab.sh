#!/bin/bash
# Gram-step split of the INT8 path (tools/lab/gram_i8_lab.cu), before and after, next to the card's name and power
# limit read in the same run.  Expects the lab binaries built for sm_100a in variants/{before,after}/gram_i8_lab_*
# (before: the parent's bnr_linalg.cu with the lab macros; see the header of gram_i8_lab.cu for the build lines).
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r3}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r3_card.txt
for b in before after; do
  for v in full loads mma bk32; do
    if [ -x variants/$b/gram_i8_lab_$v ]; then echo "## $b"; variants/$b/gram_i8_lab_$v; fi
  done
done > $OUT/r3_lab.txt 2>&1
cat $OUT/r3_card.txt $OUT/r3_lab.txt
