"""One call of each workload that goes through a different file of the engine, in this process: per call, the launch
count (psb_last_launches), a hash of every result array (CIGARs included) and, on stderr with PSB_DEBUG_TIMING=1, the
"[psb]" lines.  Run once per library build (PSB_LIB_PATH) in a fresh process and diff the outputs: after
tools/r9a_marks.py has replaced the numbers of the "[psb]" lines, both builds must print the same.
usage: PSB_DEBUG_TIMING=1 python tools/r9a_calls.py"""
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import psb_data  # noqa: E402
import parasail_rs_b200 as ps  # noqa: E402
from test_gpu_scan_routes import routed_db  # noqa: E402

FIELDS = ("score", "end_query", "end_ref", "matches", "similar", "length", "beg_query", "beg_ref", "saturated", "cigar_off", "cigar_ops")


def report(name, r):
    h = hashlib.sha1()
    for f in FIELDS:
        a = getattr(r, f)
        if a is not None:
            h.update(f.encode() + np.ascontiguousarray(a).tobytes())
    sys.stderr.flush()
    print(f"== {name}: launches {ps.launches()} n {r.n} n_retried {r.n_retried} results {h.hexdigest()[:16]}", flush=True)
    print(f"[psb] == end of {name}", file=sys.stderr, flush=True)


b62 = ps.Matrix.from_name("blosum62")
# psb_align_pairs: C1 (10^4 nw pairs of 300 x 300), C4 (10^6 sw_trace pairs of 250 x 250, over two lanes), one
# 20 kb x 20 kb sw_trace pair (traced wavefront launch and walk32), one 50 kb nw pair (wavefront)
qs, rs = psb_data.protein_pairs(1001, 10000, 300, related_frac=0.5)
report("C1 nw", ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).build().align_batch(qs, rs))
qs, rs = psb_data.protein_pairs(1004, 1000000, 250, related_frac=0.5)
report("C4 sw_trace", ps.Aligner.new().local().matrix(b62).gap_open(10).gap_extend(1).use_trace().build().align_batch(qs, rs))
del qs, rs
q = psb_data.random_seq(2001, 0, 20000)
r = psb_data.mutate(q, 2001, 1, 0.1, 0.02)[:20000]
report("20 kb sw_trace pair", ps.Aligner.new().local().matrix(b62).gap_open(10).gap_extend(1).use_trace().build().align_batch([q], [r]))
q = psb_data.random_seq(2002, 0, 50000)
r = psb_data.mutate(q, 2002, 1, 0.1, 0.02)[:50000]
report("50 kb nw pair", ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).build().align_batch([q], [r]))
# psb_align_pairs_banded: 2 000 pairs of 500 x ~510 with traceback, k = 16
qs, rs = psb_data.protein_pairs(3001, 2000, 500, related_frac=0.8, p_sub=0.1, p_indel=0.01)
report("banded nw_trace", ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).bandwidth(16).use_trace().build()
       .banded_nw_batch(qs, rs))
# psb_scan on C2 with bench.py's 400-residue query, with a query of three strips, and over routed subjects
query, cat, off = bench.make_inputs(1000000)
db = ps.Database((cat, off), b62)


def local(prof):
    return ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(prof).build()


report("C2 scan", local(ps.Profile.new(query, False, b62)).scan(db))
long_q = psb_data.random_seq(4001, 0, 1100)
report("C2 scan, 1100-residue query (3 strips)", local(ps.Profile.new(long_q, False, b62)).scan(db))
rq = psb_data.random_seq(4002, 0, 300)
rcat, roff = routed_db(4003, rq, 3, True)
report("routed subjects scan", local(ps.Profile.new(rq, False, b62)).scan(ps.Database((rcat, roff), b62)))
# psb_db_align with k = 1 000 (traceback), psb_db_subject
ids = np.random.default_rng(5).choice(len(off) - 1, 1000, replace=False)
tr = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, b62)).use_trace().build()
report("db_align k=1000", tr.align_subjects(db, ids))
h = hashlib.sha1(b"".join(np.asarray(db.subject(int(i))).tobytes() for i in ids[:50])).hexdigest()[:16]
print(f"== db_subject x 50: launches {ps.launches()} codes {h}", flush=True)
# psb_scan_host from pinned and from pageable memory
a = local(ps.Profile.new(query, False, b62))
report("scan_host pageable", a.scan_host((cat, off)))
pc = torch.empty(len(cat), dtype=torch.uint8, pin_memory=True)
pc.numpy()[:] = cat
po = torch.empty(len(off), dtype=torch.int64, pin_memory=True)
po.numpy()[:] = off
report("scan_host pinned", a.scan_host((pc.numpy(), po.numpy())))
report("scan_box 1 device", a.scan_box((pc.numpy(), po.numpy()), 1))
