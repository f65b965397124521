#!/bin/bash
# round 9a: engine.cu split into one file per path.  Parent build (variants/parent.so, built from the parent commit)
# against this tree's build: GPU suite, smoke, bench, alternating bench A/B, and one call of each workload of
# tools/r9a_calls.py per build in a fresh process: launches, result hashes and PSB_DEBUG_TIMING marks must be identical.
# usage: tools/gpu_r9a.sh OUTDIR   (reports are written under OUTDIR)
OUT=${1:?usage: tools/gpu_r9a.sh OUTDIR}
mkdir -p $OUT
BR=parasail_rs_b200/libparasail_b200.so
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > $OUT/gpu.txt
echo "devices: $(nvidia-smi -L | wc -l)" >> $OUT/gpu.txt
cat $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1; echo "build rc $?"
for v in branch parent; do
  lib=$BR; [ $v = parent ] && lib=variants/parent.so
  PSB_LIB_PATH=$PWD/$lib timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/pytest_$v.txt 2>&1
  echo "rc $?" >> $OUT/pytest_$v.txt
  echo "$v: $(tail -n 2 $OUT/pytest_$v.txt | tr '\n' ' ')"
done
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; tail -n 1 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench_1gpu.json 2> $OUT/bench_1gpu.err; tail -c 400 $OUT/bench_1gpu.json; echo
for r in 1 2 3; do timeout 600 tools/variant_bench.sh variants/parent.so $BR; done > $OUT/ab.txt 2>&1
cat $OUT/ab.txt
for v in parent branch; do
  lib=$BR; [ $v = parent ] && lib=variants/parent.so
  PSB_DEBUG_TIMING=1 PSB_LIB_PATH=$PWD/$lib timeout 900 python tools/r9a_calls.py > $OUT/calls_$v.txt 2> $OUT/calls_$v.err
  echo "rc $?" >> $OUT/calls_$v.txt
  python tools/r9a_marks.py $OUT/calls_$v.err > $OUT/marks_$v.txt
  python tools/r9a_marks.py $OUT/calls_$v.err --sorted > $OUT/marks_sorted_$v.txt
done
diff $OUT/calls_parent.txt $OUT/calls_branch.txt > $OUT/calls_diff.txt && echo "launches and results: identical" || { echo "launches or results differ"; cat $OUT/calls_diff.txt; }
diff $OUT/marks_parent.txt $OUT/marks_branch.txt > $OUT/marks_diff.txt && echo "marks: identical, in order" || echo "marks: order differs ($(wc -l < $OUT/marks_diff.txt) diff lines)"
diff $OUT/marks_sorted_parent.txt $OUT/marks_sorted_branch.txt > $OUT/marks_sorted_diff.txt && echo "marks: identical as sets per call" || { echo "marks differ per call"; head -40 $OUT/marks_sorted_diff.txt; }
cat $OUT/calls_branch.txt
echo "one device: psb_scan_box over several devices was not measured"
