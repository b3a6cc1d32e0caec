#!/bin/bash
# Outputs of the parent build (LIBBNR=variants/parent/libbnr.so) and of this tree, byte for byte, at configs 2-5;
# smoke(); the determinism check at every BASELINE shape; one kernel timeline of config 3 (tools/timeline.py) with the
# time each k_gram_slice spends beside a k_gram_i8 of another chain group.
cd "$(dirname "$0")/../.."
OUT="${OUT:-/tmp/bnr_r4}"   # where the logs go
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/r4_outputs_card.txt
Q="--steps 20 --warmup 2 --no-other-configs --no-strong --no-cpu-baseline --ess-burn 0 --ess-draws 0"
D=$(mktemp -d)
for cfg in c3 c5 c2 c4; do
  LIBBNR=$PWD/variants/parent/libbnr.so timeout 200 python bench.py $Q --config $cfg --dump-outputs $D/parent_$cfg > /dev/null 2>&1
  timeout 200 python bench.py $Q --config $cfg --dump-outputs $D/new_$cfg > /dev/null 2>&1
  n=$(ls $D/new_$cfg/*.npy | wc -l)
  if diff -r $D/parent_$cfg $D/new_$cfg > /dev/null && [ "$n" -gt 0 ]; then echo "$cfg: $n .npy files identical"
  else echo "$cfg: outputs DIFFER or missing ($n files)"; fi
done > $OUT/r4_outputs.txt
rm -rf "$D"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/r4_smoke.log 2>&1; echo "smoke rc=$?" >> $OUT/r4_smoke.log
timeout 200 python tools/timeline.py --config c3 --sweeps 2 --out $OUT/r4_timeline_c3.txt > /dev/null 2>&1
python - "$OUT/r4_timeline_c3.txt" > $OUT/r4_overlap.txt <<'PY'
import sys
rows = [l.split() for l in open(sys.argv[1]) if l[:1] != "#" and l.strip()]
ev = [(float(r[0]), float(r[2]), r[3], r[-1]) for r in rows]
sl = [e for e in ev if e[3] == "k_gram_slice"]
i8 = [e for e in ev if e[3] == "k_gram_i8"]
for s in sl:
    ov = sum(max(0.0, min(s[1], p[1]) - max(s[0], p[0])) for p in i8 if p[2] != s[2])
    print("k_gram_slice %s %8.1f us: %6.1f us beside a k_gram_i8 of another stream" % (s[2], s[1] - s[0], ov))
PY
timeout 250 bash tools/gpu_runs/r2_det.sh > $OUT/r4_det.log 2>&1
cat $OUT/r4_outputs_card.txt $OUT/r4_outputs.txt; tail -2 $OUT/r4_smoke.log; cat $OUT/r4_det.log; head -12 $OUT/r4_timeline_c3.txt; cat $OUT/r4_overlap.txt
