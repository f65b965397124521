#!/bin/bash
# round 8a: the host-memory scan split into pieces and named stages.  Parent build (variants/parent.so, built from the
# parent commit) against this tree's build: GPU suite, smoke, alternating bench A/B, and psb_scan_host's
# PSB_DEBUG_TIMING lines, launch counts, re-runs and scores on both builds, from pinned and from pageable memory
# (psb_scan_box on every device too when the box has more than one).
# usage: tools/gpu_r8a.sh OUTDIR   (reports are written under OUTDIR)
OUT=${1:?usage: tools/gpu_r8a.sh OUTDIR}
mkdir -p $OUT
BR=parasail_rs_b200/libparasail_b200.so
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader > $OUT/gpu.txt
NGPU=$(nvidia-smi -L | wc -l)
echo "devices: $NGPU" >> $OUT/gpu.txt
cat $OUT/gpu.txt
python -c "import __graft_entry__ as g; g.build()" > $OUT/build.txt 2>&1
for v in branch parent; do
  lib=$BR; [ $v = parent ] && lib=variants/parent.so
  PSB_LIB_PATH=$PWD/$lib timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider > $OUT/pytest_$v.txt 2>&1
  echo "rc $?" >> $OUT/pytest_$v.txt
  tail -n 2 $OUT/pytest_$v.txt
done
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.txt 2>&1; tail -n 1 $OUT/smoke.txt
timeout 300 python bench.py --gpus 1 --steps 5 --warmup 2 > $OUT/bench_1gpu.json 2> $OUT/bench_1gpu.err; tail -c 400 $OUT/bench_1gpu.json; echo
for r in 1 2 3; do timeout 600 tools/variant_bench.sh variants/parent.so $BR; done > $OUT/ab.txt 2>&1
cat $OUT/ab.txt
# psb_scan_host on C2, three calls in a fresh process per build and source memory: the pieces, the number of
# device-timeline marks, launches, re-runs and a hash of the results of every call
cat > $OUT/host_calls.py <<'EOF'
import hashlib, os, sys
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import numpy as np, torch, bench
import parasail_rs_b200 as ps
src, box = sys.argv[1], len(sys.argv) > 2
query, cat, off = bench.make_inputs(1000000)
if src == "pinned":
    pc = torch.empty(len(cat), dtype=torch.uint8, pin_memory=True); pc.numpy()[:] = cat
    po = torch.empty(len(off), dtype=torch.int64, pin_memory=True); po.numpy()[:] = off
    cat, off = pc.numpy(), po.numpy()
b62 = ps.Matrix.from_name("blosum62")
a = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, b62)).build()
ref = a.scan(ps.Database((cat, off), b62)) if box else None
for i in range(3):
    r = a.scan_box((cat, off), 0) if box else a.scan_host((cat, off))
    sys.stderr.flush()
    h = hashlib.sha1(np.asarray(r.score).tobytes() + np.asarray(r.end_query).tobytes() + np.asarray(r.end_ref).tobytes()).hexdigest()[:12]
    same = "" if ref is None else " equal to resident scan: " + str(all(np.array_equal(getattr(r, k), getattr(ref, k)) for k in ("score", "end_query", "end_ref")))
    print(f"== call {i}: launches {ps.launches()} n_retried {int(r.n_retried)} results {h}{same}", flush=True)
EOF
summarise() {   # one run's output -> per call: its pieces lines, its number of device-timeline marks, launches / re-runs / hash
  python - "$1" <<'EOF'
import re, sys
for line in open(sys.argv[1]):
    if "pieces (MB)" in line:
        print(re.sub(r"; upload .*", "", line.strip()))
    elif "device timeline" in line:
        print(line.split(": device")[0], "marks", len(line.split("entry):")[1].split()))
    elif line.startswith("=="):
        print(line.strip())
EOF
}
first() { awk '{print} /== call 0/{exit}' $1; }
runs="pinned pageable"
[ "$NGPU" -gt 1 ] && runs="$runs box"
for src in $runs; do
  for v in parent branch; do
    lib=$BR; [ $v = parent ] && lib=variants/parent.so
    arg=$src; extra=; [ $src = box ] && { arg=pinned; extra=box; }
    PSB_DEBUG_TIMING=1 PSB_LIB_PATH=$PWD/$lib timeout 600 python $OUT/host_calls.py $arg $extra > $OUT/host_${src}_$v.txt 2>&1
    echo "rc $?" >> $OUT/host_${src}_$v.txt
    summarise $OUT/host_${src}_$v.txt > $OUT/host_${src}_$v.sum
  done
  # the first call uses default rates: its pieces, marks, launches, re-runs and results must match; later calls are reported
  diff <(first $OUT/host_${src}_parent.sum) <(first $OUT/host_${src}_branch.sum) > $OUT/host_${src}_first_diff.txt \
    && echo "$src: first call identical" || { echo "$src: first call differs"; cat $OUT/host_${src}_first_diff.txt; }
  diff <(grep "==\|marks" $OUT/host_${src}_parent.sum) <(grep "==\|marks" $OUT/host_${src}_branch.sum) > $OUT/host_${src}_all_diff.txt \
    && echo "$src: marks, launches, re-runs and results of all calls identical" || { echo "$src: later calls differ"; cat $OUT/host_${src}_all_diff.txt; }
  for v in parent branch; do echo "-- $src $v"; cat $OUT/host_${src}_$v.sum; done
done
if [ "$NGPU" -gt 1 ]; then
  for N in 2 4 8; do
    [ $N -gt $NGPU ] && continue
    for v in parent branch; do
      lib=$BR; [ $v = parent ] && lib=variants/parent.so
      PSB_LIB_PATH=$PWD/$lib timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 2971$N \
        bench.py --gpus $N --steps 10 --warmup 3 --e2e-steps 10 > $OUT/bench_${N}gpu_$v.json 2> $OUT/bench_${N}gpu_$v.err
      python -c "
import json; d=json.load(open('$OUT/bench_${N}gpu_$v.json')); print('$v N', d['n_gpus'], 'value', round(d['value']), 'e2e', round(d['e2e']['value']), (d['config'].get('verified') or '')[:60])"
    done
  done
else
  echo "one device: the multi-GPU path (psb_scan_box over several devices) was not measured"
fi
