#!/bin/bash
# k_gram_slice, new (launch_gram_slice) against the previous kernel kept in the lab (k_gram_slice_ref): planes and row
# scales byte for byte on the check inputs, then both timed in the full build and in the two diagnostic builds (no plane
# stores, no digit math), next to the card's name and power limit read in the same run.  Expects the lab binaries built
# for sm_100a in variants/after/gram_i8_lab_{full,nostore,nodigit} (build lines in the header of gram_i8_lab.cu).
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r4}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r4_card.txt
timeout 300 variants/after/gram_i8_lab_full check > $OUT/r4_check.txt 2>&1; echo "check rc=$?" >> $OUT/r4_check.txt
for v in full nostore nodigit; do timeout 120 variants/after/gram_i8_lab_$v; done > $OUT/r4_lab.txt 2>&1
cat $OUT/r4_card.txt $OUT/r4_check.txt $OUT/r4_lab.txt
