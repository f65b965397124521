#!/bin/bash
# round 11a: a resident database sharded over the box (BoxDatabase, psb_box_*).  The new GPU tests, the whole GPU suite,
# smoke, bench, and tools/box_search_probe.py (box against one device, on 1 / 2 / 4 / 8 visible GPUs).
# usage: tools/gpu_r11a.sh OUTDIR   (reports are written under OUTDIR)
OUT=${1:?usage: tools/gpu_r11a.sh OUTDIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/gpu.txt
cat $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1; echo "build rc $?"
timeout 900 python -m pytest tests/test_gpu_box_search.py -q -p no:cacheprovider -rs > $OUT/pytest_box_search.txt 2>&1
echo "rc $?" >> $OUT/pytest_box_search.txt; tail -n 30 $OUT/pytest_box_search.txt
timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider --ignore=tests/test_gpu_box_search.py > $OUT/pytest_gpu.txt 2>&1
echo "rc $?" >> $OUT/pytest_gpu.txt; tail -n 4 $OUT/pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; tail -n 1 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench_1gpu.json 2> $OUT/bench_1gpu.err; tail -c 400 $OUT/bench_1gpu.json; echo
timeout 900 python tools/box_search_probe.py --reps 3 --out $OUT/box_search_probe.json > $OUT/box_search_probe.txt 2>&1; echo "probe rc $?"
grep '^N=\|^{' $OUT/box_search_probe.txt | cut -c1-600 | head -n 12
