#!/bin/bash
# round 10a: many queries in one call (psb_db_search).  The new GPU tests, the whole GPU suite, smoke, bench, and
# tools/search_probe.py (psb_db_search against the per-query composition it replaces).
# usage: tools/gpu_r10a.sh OUTDIR   (reports are written under OUTDIR)
OUT=${1:?usage: tools/gpu_r10a.sh OUTDIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > $OUT/gpu.txt
cat $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1; echo "build rc $?"
timeout 900 python -m pytest tests/test_gpu_search_many.py -q -p no:cacheprovider > $OUT/pytest_search_many.txt 2>&1
echo "rc $?" >> $OUT/pytest_search_many.txt; tail -n 30 $OUT/pytest_search_many.txt
timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/pytest_gpu.txt 2>&1
echo "rc $?" >> $OUT/pytest_gpu.txt; tail -n 4 $OUT/pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; tail -n 1 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench_1gpu.json 2> $OUT/bench_1gpu.err; tail -c 400 $OUT/bench_1gpu.json; echo
timeout 900 python tools/search_probe.py --out $OUT/search_probe.json > $OUT/search_probe.txt 2>&1; echo "probe rc $?"
grep -v '^ \|^{\|^}' $OUT/search_probe.txt | tail -n 12
