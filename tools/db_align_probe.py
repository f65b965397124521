#!/usr/bin/env python
"""What aligning the hits of a scan costs on the C2-size resident database (psb_db_align).

usage: python tools/db_align_probe.py [--db 1000000] [--reps 7] [--out FILE.json]

One 400-aa query (bench.py's) against the resident database of bench.py's synthetic proteins, BLOSUM62 10/1.
Per case: kernel ms (psb_last_kernel_ms), wall ms of the call ending in a device synchronise, and launches, the
median over --reps calls after a warm-up:
  scan             psb_scan, sw_striped_profile_sat (the score-only scan search() starts with)
  search k         Aligner.search(db, k) with sw_trace: scan + top-k + psb_db_align of the k hits
  align k          psb_db_align of the same k ids alone
  stats all        psb_db_align with sw_stats over every subject, next to psb_scan with the same name
For each k also the library's PSB_DEBUG_TIMING lines of one more call (kernel times and host phases of the pass)
and the longest / median number of cells a hit's traceback walk visits.
Checked inside the run: every hit's CIGAR re-scores to its score and lands on its end cell, every hit's
(score, end_query, end_ref) equals the scan's, and the _stats batch equals psb_scan's on all six fields.
The card's name and power limit are read in the same run and written beside the figures.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import bench  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "error": repr(e)}


def timed(ps, fn, reps):
    fn()
    rows = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ps._lib.lib().psb_synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        rows.append((wall, ps.kernel_ms(), ps.launches()))
    med = lambda i: statistics.median(r[i] for r in rows)
    return out, {"wall_ms": round(med(0), 3), "kernel_ms": round(med(1), 3), "launches": int(med(2)),
                 "wall_ms_min": round(min(r[0] for r in rows), 3)}


def debug_timing(fn):
    """the library's PSB_DEBUG_TIMING lines (host phases and kernel times of each pass) of one call of fn"""
    import tempfile
    with tempfile.TemporaryFile(mode="w+") as tf:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(tf.fileno(), 2)
        os.environ["PSB_DEBUG_TIMING"] = "1"
        try:
            fn()
        finally:
            del os.environ["PSB_DEBUG_TIMING"]
            os.dup2(saved, 2)
            os.close(saved)
        tf.seek(0)
        return [" ".join(line.split()) for line in tf if line.startswith("[psb]")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from __graft_entry__ import build
    build()
    import parasail_rs_b200 as ps
    from oracle import oracle as orc
    import psb_data

    query, cat, off = bench.make_inputs(args.db)
    b62 = ps.Matrix.from_name("blosum62")
    omat = orc.Matrix.from_table(psb_data.BLOSUM62_ALPHABET, psb_data.blosum62_table())
    db = ps.Database((cat, off), b62)
    prof = ps.Profile.new(query, False, b62)
    mk = lambda: ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(prof)
    scan_a, trace_a = mk().build(), mk().use_trace().build()
    lq = len(query)
    res = {"workload": f"one {lq}-aa query vs {args.db} synthetic proteins ({int(off[-1])} residues, bench.py's seeds), "
                       f"BLOSUM62 open {bench.OPEN} ext {bench.GAP}, local", "reps": args.reps, **card(), "cases": {}}

    scan, res["cases"]["scan"] = timed(ps, lambda: scan_a.scan(db), args.reps)
    res["cases"]["scan"]["cells"] = float(lq) * float(off[-1])
    for k in (100, 1000, 10000):
        (ids, hits), res["cases"][f"search {k}"] = timed(ps, lambda: trace_a.search(db, k), args.reps)
        _, res["cases"][f"align {k}"] = timed(ps, lambda: trace_a.align_subjects(db, ids), args.reps)
        rc, ro = psb_data.concat([cat[off[i]:off[i + 1]] for i in ids])
        res["cases"][f"align {k}"]["cells"] = float(lq) * float(ro[-1])
        res["cases"][f"align {k}"]["cigar_words"] = int(hits.cigar_off[-1])
        # cells each hit's traceback walk visits (sum of its CIGAR run lengths): the walk is one thread per pair
        path = np.add.reduceat((hits.cigar_ops >> 4).astype(np.int64), hits.cigar_off[:-1])
        res["cases"][f"align {k}"]["walk_cells_max_median"] = [int(path.max()), int(np.median(path))]
        res["cases"][f"align {k}"]["debug_timing"] = debug_timing(lambda: trace_a.align_subjects(db, ids))
        for f in ("score", "end_query", "end_ref"):
            assert np.array_equal(getattr(hits, f), getattr(scan, f)[ids]), (k, f)
        qcat, qoff = np.tile(query, len(ids)), np.arange(len(ids) + 1, dtype=np.int64) * lq
        bad, first = orc.cigar_check_batch(qcat, qoff, rc, ro, omat, 2, bench.OPEN, bench.GAP, hits.cigar_ops, hits.cigar_off,
                                           hits.beg_query, hits.beg_ref, hits.end_query, hits.end_ref, hits.score)
        assert bad == 0, f"k={k}: {bad} CIGARs do not re-score, first at {first}"
        res["cases"][f"search {k}"]["checked"] = "CIGARs re-score to the score and end cell; hits equal the scan"
        res["cases"][f"search {k}"]["note"] = "wall: the whole search; kernel_ms / launches: its psb_db_align call (the scan's are under scan)"

    sprof = ps.Profile.new(query, True, b62)
    stats_a = ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(sprof).build()
    got, res["cases"]["stats all: psb_db_align"] = timed(ps, lambda: stats_a.align_subjects(db), args.reps)
    ref, res["cases"]["stats all: psb_scan"] = timed(ps, lambda: stats_a.scan(db), args.reps)
    for f in ("score", "end_query", "end_ref", "matches", "similar", "length"):
        assert np.array_equal(getattr(got, f), getattr(ref, f)), f
    res["cases"]["stats all: psb_db_align"]["checked"] = "equal to psb_scan on all six fields"

    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
