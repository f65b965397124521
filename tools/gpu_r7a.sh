#!/bin/bash
# round 7a: the database scan's host side split into a plan and stages.  Parent build (variants/parent.so, built from the
# parent commit) against this tree's build: GPU suite, smoke, alternating bench A/B, and the scan's PSB_DEBUG_TIMING
# lines and launch counts on both builds.
# usage: tools/gpu_r7a.sh OUTDIR   (reports are written under OUTDIR)
OUT=${1:?usage: tools/gpu_r7a.sh OUTDIR}
mkdir -p $OUT
BR=parasail_rs_b200/libparasail_b200.so
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1
for v in branch parent; do
  lib=$BR; [ $v = parent ] && lib=variants/parent.so
  PSB_LIB_PATH=$PWD/$lib timeout 600 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/pytest_$v.txt 2>&1
  echo "rc $?" >> $OUT/pytest_$v.txt
  tail -n 2 $OUT/pytest_$v.txt
done
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; tail -n 1 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench_1gpu.json 2> $OUT/bench_1gpu.err; tail -c 400 $OUT/bench_1gpu.json
for r in 1 2 3; do timeout 600 tools/variant_bench.sh variants/parent.so $BR; done > $OUT/ab.txt 2>&1
cat $OUT/ab.txt
# scan_sw16's stages: C2-sized single strip (head), a 1000 aa query (strips), a 70 kb subject (route); the re-run launch is in every count
for v in parent branch; do
  lib=$BR; [ $v = parent ] && lib=variants/parent.so
  PSB_DEBUG_TIMING=1 PSB_LIB_PATH=$PWD/$lib timeout 600 python - > $OUT/stages_$v.txt 2>&1 <<'EOF'
import os, sys
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import hashlib
import numpy as np, psb_data
import parasail_rs_b200 as ps
b62 = ps.Matrix.from_name("blosum62")
cat, off = psb_data.protein_db(2002, 2003, 200000)
big = np.concatenate([cat, np.frombuffer(bytes(psb_data.random_seq(7, 0, 70000)), dtype=np.uint8)])
boff = np.concatenate([off, [off[-1] + 70000]]).astype(np.int64)
for name, (c, o) in (("c2", (cat, off)), ("c2+70kb", (big, boff))):
    db = ps.Database((c, o), b62)
    for lq in (400, 1000):
        q = psb_data.random_seq(2001, 0, lq)
        a = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(q, False, b62)).build()
        for _ in range(2):
            r = a.scan(db)
        print(f"== {name} lq {lq}: launches {ps.launches()} n_retried {int(r.n_retried)} scores {hashlib.sha1(np.asarray(r.score).tobytes()).hexdigest()[:12]}", flush=True)
EOF
  grep -v "scan job" $OUT/stages_$v.txt | grep "==\|sw16" | sed 's/est [0-9.]* ms long_len [0-9]* //' > $OUT/stages_$v.cmp
done
diff $OUT/stages_parent.cmp $OUT/stages_branch.cmp > $OUT/stages_diff.txt && echo "stage lines identical" || { echo "stage lines differ"; head -20 $OUT/stages_diff.txt; }
cat $OUT/stages_branch.cmp
